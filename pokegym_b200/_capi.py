"""ctypes binding of the C ABI declared in include/gbenv.h.

The product loads ``pokegym_b200/csrc/libgbenv.so`` (prefix ``gbenv_``) and nothing else; when that
library is missing the import of :mod:`pokegym_b200.vec_env` fails loudly -- there is no CPU fallback.
The same binding class is reused by the tests to drive the CPU oracle (prefix ``oracle_``), which
implements the identical entry points over host memory.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

import numpy as np

STATE_BYTES = 142_610
OBS_H, OBS_W, OBS_C = 72, 80, 4
OBS_BYTES = OBS_H * OBS_W * OBS_C
INFO_SCALARS = 72
ABI_VERSION = 9
COUNTS_H, COUNTS_W = 444, 436
SCREEN_H, SCREEN_W = 144, 160
FRAME_WORDS = 1440  # packed frame: 144 lines x 10 uint32 words of 16 2-bit shades (include/gbenv.h)
EVENT_FLAGS = 130  # entries of the reference's event table (pokegym_b200/event_table.json)
EVENT_WORDS = 5  # uint32 words of one env's event flags
OBS_PACKED_WORDS = 576  # packed observation: 72 rows x 8 uint32 words, 3 bits per pixel (include/gbenv.h)
OBS_PACKED_BYTES = OBS_PACKED_WORDS * 4
NUM_ACTIONS = 8
ACT_FREQ = 24

PKG_DIR = Path(__file__).resolve().parent
DEFAULT_LIB = PKG_DIR / "csrc" / "libgbenv.so"


class Counters(C.Structure):
    _fields_ = [("instructions", C.c_uint64), ("cycles", C.c_uint64), ("frames", C.c_uint64), ("faults", C.c_uint64),
                ("kernel_launches", C.c_uint64)]


class CoreExtra(C.Structure):
    _fields_ = [("stat_mode", C.c_int32), ("ly_window", C.c_int32), ("fault", C.c_int32), ("reserved", C.c_int32)]


class GbEnvError(RuntimeError):
    pass


def _ptr(x) -> C.c_void_p:
    """Device/host pointer of a torch tensor, numpy array, int address or None."""
    if x is None:
        return C.c_void_p(0)
    if isinstance(x, int):
        return C.c_void_p(x)
    if isinstance(x, np.ndarray):
        if not x.flags["C_CONTIGUOUS"]:
            raise ValueError("array must be C-contiguous")
        return C.c_void_p(x.ctypes.data)
    if hasattr(x, "data_ptr"):
        return C.c_void_p(x.data_ptr())
    raise TypeError(f"cannot take the address of {type(x)}")


def _nbytes(x) -> int:
    """Size in bytes of a torch tensor or numpy array."""
    return int(x.numel() * x.element_size()) if hasattr(x, "element_size") else int(x.nbytes)


def _byte_rows(x, row_bytes: int, what: str, n=None) -> int:
    """Number of rows of `x`, a C-contiguous, 16-byte aligned uint8 torch tensor or numpy array of whole `row_bytes` rows
    (exactly `n` of them when given).  Raw pointers cross the C ABI, so a wrong buffer would be out-of-bounds writes."""
    if isinstance(x, np.ndarray):
        ok, addr = x.dtype == np.uint8 and x.flags["C_CONTIGUOUS"], x.ctypes.data
    elif hasattr(x, "data_ptr"):
        ok, addr = str(x.dtype) == "torch.uint8" and x.is_contiguous(), x.data_ptr()
    else:
        raise TypeError(f"{what} must be a torch tensor or numpy array, not {type(x)}")
    size = _nbytes(x)
    if not ok or addr % 16 or size % row_bytes or (n is not None and size != n * row_bytes):
        rows = "whole" if n is None else str(n)
        raise ValueError(f"{what} must be a contiguous, 16-byte aligned uint8 buffer of {rows} rows of {row_bytes} bytes")
    return size // row_bytes


# name -> (argtypes, restype); shared by both libraries
_SIGS = {
    "abi_version": ([], C.c_int),
    "create": ([C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)], C.c_int),
    "destroy": ([C.c_void_p], C.c_int),
    "last_error": ([C.c_void_p], C.c_char_p),
    "num_envs": ([C.c_void_p], C.c_int),
    "sync": ([C.c_void_p], C.c_int),
    "check": ([C.c_void_p], C.c_int),
    "set_lanes_per_warp": ([C.c_void_p, C.c_int], C.c_int),
    "get_lanes_per_warp": ([C.c_void_p], C.c_int),
    "add_state_template": ([C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)], C.c_int),
    "load_template": ([C.c_void_p, C.c_void_p, C.c_int, C.c_int], C.c_int),
    "set_initial_template": ([C.c_void_p, C.c_void_p, C.c_int, C.c_int], C.c_int),
    "power_on": ([C.c_void_p, C.c_void_p, C.c_int], C.c_int),
    "save_state": ([C.c_void_p, C.c_int, C.c_void_p], C.c_int),
    "save_states": ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p], C.c_int),
    "load_states": ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "run_action": ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p], C.c_int),
    "tick": ([C.c_void_p, C.c_int, C.c_int, C.c_void_p], C.c_int),
    "send_input": ([C.c_void_p, C.c_int, C.c_int, C.c_void_p], C.c_int),
    "read_mem": ([C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_void_p], C.c_int),
    "write_mem": ([C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_void_p], C.c_int),
    "screen": ([C.c_void_p, C.c_int, C.c_void_p], C.c_int),
    "capture_frames": ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p], C.c_int),
    "frames_to_rgb": ([C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p], C.c_int),
    "event_flags": ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p], C.c_int),
    "reset": ([C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p], C.c_int),
    "reset_dev": ([C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p], C.c_int),
    "submit_host": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "fetch_host": ([C.c_void_p], C.c_int),
    "step": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "step_masked": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "step_packed": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "reset_packed": ([C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p], C.c_int),
    "unpack_obs": ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p], C.c_int),
    "step_host": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "reset_host": ([C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p], C.c_int),
    "get_info": ([C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "reduce_info": ([C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "reduce_info_masked": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "counts_map": ([C.c_void_p, C.c_int, C.c_void_p], C.c_int),
    "counts_map_sum": ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p], C.c_int),
    "get_counters": ([C.c_void_p, C.POINTER(Counters)], C.c_int),
    "last_kernel_ms": ([C.c_void_p, C.c_int, C.POINTER(C.c_float)], C.c_int),
    "kernel_time_total": ([C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_uint64)], C.c_int),
    "get_core_extra": ([C.c_void_p, C.c_int, C.POINTER(CoreExtra)], C.c_int),
    "debug_render_frame": ([C.c_void_p, C.c_int], C.c_int),
}

EXPORTED_SYMBOLS = tuple(_SIGS)


class GbEnvLib:
    """Loaded shared library implementing the gbenv ABI."""

    def __init__(self, path: os.PathLike, prefix: str = "gbenv_"):
        self.path = str(path)
        self.prefix = prefix
        if not Path(self.path).exists():
            raise GbEnvError(
                f"{self.path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                f"(there is no CPU fallback for the CUDA library)"
            )
        self.dll = C.CDLL(self.path)
        for name, (argtypes, restype) in _SIGS.items():
            fn = getattr(self.dll, prefix + name)
            fn.argtypes = argtypes
            fn.restype = restype
            setattr(self, name, fn)
        if self.abi_version() != ABI_VERSION:  # buffer sizes (info row width) are fixed by the ABI version
            raise GbEnvError(f"{self.path}: ABI version {self.abi_version()} != {ABI_VERSION} expected by this package; rebuild the library")


class Handle:
    """Owning wrapper of a ``gbenv_t*`` with error-code checking."""

    def __init__(self, lib: GbEnvLib, n_envs: int, rom: bytes, device_id: int = 0):
        self.lib = lib
        self.n_envs = int(n_envs)
        self._h = C.c_void_p(0)
        rom_buf = (C.c_uint8 * len(rom)).from_buffer_copy(rom)
        rc = lib.create(self.n_envs, C.cast(rom_buf, C.c_void_p), len(rom), int(device_id), C.byref(self._h))
        if rc != 0:
            msg = lib.last_error(None)
            raise GbEnvError(f"{lib.prefix}create failed ({rc}): {msg.decode() if msg else ''}")

    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self.lib.last_error(self._h)
            raise GbEnvError(f"{self.lib.prefix}{what} failed ({rc}): {msg.decode() if msg else ''}")

    def close(self):
        if self._h:
            self.lib.destroy(self._h)
            self._h = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- templates / state ---------------------------------------------------
    @staticmethod
    def _ids(env_ids):
        if env_ids is None:
            return C.c_void_p(0), 0, None
        a = np.ascontiguousarray(env_ids, dtype=np.int32)
        return C.c_void_p(a.ctypes.data), int(a.size), a

    def add_state_template(self, blob: bytes) -> int:
        tid = C.c_int(-1)
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        self._check(self.lib.add_state_template(self._h, C.cast(buf, C.c_void_p), len(blob), C.byref(tid)), "add_state_template")
        return tid.value

    def load_template(self, template_id: int, env_ids=None):
        p, n, keep = self._ids(env_ids)
        self._check(self.lib.load_template(self._h, p, n, int(template_id)), "load_template")

    def set_initial_template(self, template_id: int, env_ids=None):
        p, n, keep = self._ids(env_ids)
        self._check(self.lib.set_initial_template(self._h, p, n, int(template_id)), "set_initial_template")

    def power_on(self, env_ids=None):
        p, n, keep = self._ids(env_ids)
        self._check(self.lib.power_on(self._h, p, n), "power_on")

    def save_state(self, env: int) -> bytes:
        out = np.empty(STATE_BYTES, dtype=np.uint8)
        self._check(self.lib.save_state(self._h, int(env), _ptr(out)), "save_state")
        return out.tobytes()

    def save_states(self, out, env_ids=None, stream=None):
        """The v9 .state file of the envs `env_ids` (int32, on the device for CUDA, host memory for the oracle; None: envs
        0..len(out)-1) -> out uint8 [n, STATE_BYTES], each row what save_state() returns for its env.  Rows of ids outside
        [0, n_envs) are left untouched."""
        n = _byte_rows(out, STATE_BYTES, "out", None if env_ids is None else len(env_ids))
        self._check(self.lib.save_states(self._h, _ptr(env_ids), int(n), _ptr(out), C.c_void_p(stream or 0)), "save_states")

    def load_states(self, blobs, env_ids=None, status=None, stream=None):
        """PyBoy.load_state of row i of blobs uint8 [n, STATE_BYTES] into env env_ids[i] (int32, on the device for CUDA, host
        memory for the oracle; None: envs 0..n-1).  status (int32 [n], or None) gets 0 for a loaded row, GBENV_E_STATE (-2)
        for a rejected one and GBENV_E_ARG (-1) for an id outside [0, n_envs), whose row is skipped."""
        n = _byte_rows(blobs, STATE_BYTES, "blobs", None if env_ids is None else len(env_ids))
        if status is not None:
            if isinstance(status, np.ndarray):
                ok = status.dtype == np.int32 and status.flags["C_CONTIGUOUS"]
            else:
                ok = str(status.dtype) == "torch.int32" and status.is_contiguous()
            if not ok or _nbytes(status) != 4 * n:
                raise ValueError(f"status must be a contiguous int32 buffer of {n} entries")
        self._check(self.lib.load_states(self._h, _ptr(env_ids), int(n), _ptr(blobs), _ptr(status), C.c_void_p(stream or 0)), "load_states")

    # -- emulator ------------------------------------------------------------
    def run_action(self, actions, frame_skip: int = ACT_FREQ, stream: int = 0):
        self._check(self.lib.run_action(self._h, _ptr(actions), int(frame_skip), C.c_void_p(stream)), "run_action")

    def tick(self, n_frames: int = 1, render: bool = True, stream: int = 0):
        self._check(self.lib.tick(self._h, int(n_frames), int(bool(render)), C.c_void_p(stream)), "tick")

    def send_input(self, button: int, pressed: bool, stream: int = 0):
        self._check(self.lib.send_input(self._h, int(button), int(bool(pressed)), C.c_void_p(stream)), "send_input")

    def read_mem(self, env: int, addr: int, n: int = 1) -> np.ndarray:
        out = np.empty(n, dtype=np.uint8)
        self._check(self.lib.read_mem(self._h, int(env), int(addr), int(n), _ptr(out)), "read_mem")
        return out

    def write_mem(self, env: int, addr: int, data):
        a = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        self._check(self.lib.write_mem(self._h, int(env), int(addr), int(a.size), _ptr(a)), "write_mem")

    def screen(self, env: int) -> np.ndarray:
        out = np.empty((144, 160, 3), dtype=np.uint8)
        self._check(self.lib.screen(self._h, int(env), _ptr(out)), "screen")
        return out

    def capture_frames(self, frames, env_ids=None, stream: int = 0):
        """The current packed frame of the envs `env_ids` (int32, on the device for CUDA, host memory for the oracle; None:
        envs 0..len(frames)-1) -> frames uint32 [n, FRAME_WORDS].  Rows of ids outside [0, n_envs) are left untouched."""
        n = len(frames) if env_ids is None else len(env_ids)
        if _nbytes(frames) < n * FRAME_WORDS * 4:
            raise ValueError(f"frames holds fewer than {n} packed frames")
        self._check(self.lib.capture_frames(self._h, _ptr(env_ids), int(n), _ptr(frames), C.c_void_p(stream)), "capture_frames")

    def frames_to_rgb(self, frames, out, channels: int = 3, stream: int = 0):
        """Packed frames uint32 [n, FRAME_WORDS] -> out uint8 [n, 144, 160, channels] (1 = grey, 3 = RGB as screen())."""
        if _nbytes(frames) < len(frames) * FRAME_WORDS * 4 or _nbytes(out) < len(frames) * SCREEN_H * SCREEN_W * max(int(channels), 0):
            raise ValueError("frames must be [n, FRAME_WORDS] words and out must hold n decoded frames")
        self._check(self.lib.frames_to_rgb(self._h, _ptr(frames), int(len(frames)), int(channels), _ptr(out), C.c_void_p(stream)),
                    "frames_to_rgb")

    def event_flags(self, out, env_ids=None, stream: int = 0):
        """The event flags of the envs `env_ids` (int32, on the device for CUDA, host memory for the oracle; None: envs
        0..len(out)-1) -> out uint32 [n, EVENT_WORDS]: bit k & 31 of word k >> 5 is entry k of the event table.  Rows of ids
        outside [0, n_envs) are left untouched."""
        n = len(out) if env_ids is None else len(env_ids)
        if _nbytes(out) < n * EVENT_WORDS * 4:
            raise ValueError(f"out holds fewer than {n} rows of event flags")
        self._check(self.lib.event_flags(self._h, _ptr(env_ids), int(n), _ptr(out), C.c_void_p(stream)), "event_flags")

    # -- Environment API -----------------------------------------------------
    def reset(self, obs, mask=None, max_episode_steps: int = 20480, reward_scale: float = 4.0, obs_stride: int = OBS_BYTES, stream: int = 0):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        self._check(
            self.lib.reset(self._h, _ptr(m), int(max_episode_steps), float(reward_scale), _ptr(obs), int(obs_stride), C.c_void_p(stream)),
            "reset",
        )

    def reset_dev(self, obs, mask_dev=None, max_episode_steps: int = 20480, reward_scale: float = 4.0, obs_stride: int = OBS_BYTES, stream: int = 0):
        """Environment.reset for the envs whose byte in the DEVICE mask is non-zero (None: all); nothing touches the host."""
        self._check(
            self.lib.reset_dev(self._h, _ptr(mask_dev), int(max_episode_steps), float(reward_scale), _ptr(obs), int(obs_stride), C.c_void_p(stream)),
            "reset_dev",
        )

    def submit_host(self, actions: np.ndarray, obs: np.ndarray, reward: np.ndarray, done: np.ndarray):
        self._check(self.lib.submit_host(self._h, _ptr(actions), _ptr(obs), _ptr(reward), _ptr(done)), "submit_host")

    def fetch_host(self):
        self._check(self.lib.fetch_host(self._h), "fetch_host")

    def step(self, actions, obs, reward, done, obs_stride: int = OBS_BYTES, stream: int = 0):
        self._check(self.lib.step(self._h, _ptr(actions), _ptr(obs), int(obs_stride), _ptr(reward), _ptr(done), C.c_void_p(stream)), "step")

    def step_masked(self, actions, skip, obs, reward, done, obs_stride: int = OBS_BYTES, stream: int = 0):
        """Environment.step for the envs with skip[e] == 0; the others sit the step out (reward 0, done 0, obs row untouched)."""
        self._check(self.lib.step_masked(self._h, _ptr(actions), _ptr(skip), _ptr(obs), int(obs_stride), _ptr(reward), _ptr(done), C.c_void_p(stream)),
                    "step_masked")

    def step_packed(self, actions, skip, packed, reward, done, stream: int = 0):
        """step_masked with the observation packed: packed uint8 [n_envs, OBS_PACKED_BYTES] (rows of skipped envs untouched)."""
        _byte_rows(packed, OBS_PACKED_BYTES, "packed", self.n_envs)
        self._check(self.lib.step_packed(self._h, _ptr(actions), _ptr(skip), _ptr(packed), _ptr(reward), _ptr(done), C.c_void_p(stream)),
                    "step_packed")

    def reset_packed(self, packed, mask_dev=None, max_episode_steps: int = 20480, reward_scale: float = 4.0, stream: int = 0):
        """reset_dev with the observation packed: packed uint8 [n_envs, OBS_PACKED_BYTES], only the reset envs' rows written."""
        _byte_rows(packed, OBS_PACKED_BYTES, "packed", self.n_envs)
        self._check(self.lib.reset_packed(self._h, _ptr(mask_dev), int(max_episode_steps), float(reward_scale), _ptr(packed), C.c_void_p(stream)),
                    "reset_packed")

    def unpack_obs(self, packed, out, stream: int = 0):
        """Packed rows uint8 [n, OBS_PACKED_BYTES] -> out uint8 [n, OBS_BYTES], the reference observations."""
        n = _byte_rows(packed, OBS_PACKED_BYTES, "packed")
        _byte_rows(out, OBS_BYTES, "out", n)
        self._check(self.lib.unpack_obs(self._h, _ptr(packed), n, _ptr(out), C.c_void_p(stream)), "unpack_obs")

    def step_host(self, actions: np.ndarray, obs: np.ndarray, reward: np.ndarray, done: np.ndarray):
        self._check(self.lib.step_host(self._h, _ptr(actions), _ptr(obs), _ptr(reward), _ptr(done)), "step_host")

    def reset_host(self, obs: np.ndarray, mask=None, max_episode_steps: int = 20480, reward_scale: float = 4.0):
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        self._check(self.lib.reset_host(self._h, _ptr(m), int(max_episode_steps), float(reward_scale), _ptr(obs)), "reset_host")

    def get_info(self, info, stream: int = 0):
        self._check(self.lib.get_info(self._h, _ptr(info), C.c_void_p(stream)), "get_info")

    def reduce_info(self, out, stream: int = 0):
        self._check(self.lib.reduce_info(self._h, _ptr(out), C.c_void_p(stream)), "reduce_info")

    def reduce_info_masked(self, out, mask_dev=None, stream: int = 0):
        """reduce_info over the envs whose mask byte is non-zero (None: all); slot 0 = how many of them have stepped."""
        self._check(self.lib.reduce_info_masked(self._h, _ptr(mask_dev), _ptr(out), C.c_void_p(stream)), "reduce_info_masked")

    def counts_map(self, env: int) -> np.ndarray:
        out = np.empty((COUNTS_H, COUNTS_W), dtype=np.int32)
        self._check(self.lib.counts_map(self._h, int(env), _ptr(out)), "counts_map")
        return out

    def counts_map_sum(self, out, mask_dev=None, stream: int = 0):
        """int64 [444, 436] sum of the heat maps of the envs whose mask byte is non-zero (None: all) -> out (overwritten)."""
        self._check(self.lib.counts_map_sum(self._h, _ptr(mask_dev), _ptr(out), C.c_void_p(stream)), "counts_map_sum")

    # -- diagnostics ---------------------------------------------------------
    def sync(self):
        self._check(self.lib.sync(self._h), "sync")

    def check(self):
        """sync + raise if a pool of the exploration storage (visited bitmaps / heat maps) ran dry"""
        self._check(self.lib.check(self._h), "check")

    def lanes_per_warp(self) -> int:
        return int(self.lib.get_lanes_per_warp(self._h))

    def set_lanes_per_warp(self, lanes: int):
        self._check(self.lib.set_lanes_per_warp(self._h, int(lanes)), "set_lanes_per_warp")

    def counters(self) -> Counters:
        c = Counters()
        self._check(self.lib.get_counters(self._h, C.byref(c)), "get_counters")
        return c

    def last_kernel_ms(self, which: int = 0) -> float:
        ms = C.c_float(0)
        self._check(self.lib.last_kernel_ms(self._h, int(which), C.byref(ms)), "last_kernel_ms")
        return ms.value

    def kernel_time_total(self, which: int = 0):
        """(total device ms, steps) of kernel group `which` (0 = emulate, 1 = reward + obs) since create."""
        ms, steps = C.c_double(0), C.c_uint64(0)
        self._check(self.lib.kernel_time_total(self._h, int(which), C.byref(ms), C.byref(steps)), "kernel_time_total")
        return ms.value, steps.value

    def debug_render_frame(self, env: int):
        self._check(self.lib.debug_render_frame(self._h, int(env)), "debug_render_frame")

    def core_extra(self, env: int) -> CoreExtra:
        x = CoreExtra()
        self._check(self.lib.get_core_extra(self._h, int(env), C.byref(x)), "get_core_extra")
        return x
