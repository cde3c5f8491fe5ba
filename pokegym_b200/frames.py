"""Full-resolution frames of chosen envs, kept on the device: the frames the reference's `save_video` / `fast_video` writes
and `render()` shows (pyboy_binding.py:77-78,86-87), for a batch.

Frames are stored PACKED, as the library keeps the framebuffer (include/gbenv.h, GBENV_FRAME_WORDS): 1,440 uint32 words,
2 bits per pixel, 5,760 B per frame, 12x smaller than RGB and lossless.  They are expanded to grey or RGB only on request,
on the device (gbenv_frames_to_rgb).  Writing video files is left to the caller.
"""
from __future__ import annotations

import numpy as np

from . import _capi

FRAME_SHAPE = (_capi.SCREEN_H, _capi.SCREEN_W)


def host_env_ids(env_ids, num_envs: int) -> np.ndarray:
    """env_ids as a 1-D int32 host array, every id in [0, num_envs).  Raw pointers cross the C ABI, so ids are checked here
    rather than trusted; a device tensor is copied to the host for the check."""
    if hasattr(env_ids, "detach"):
        env_ids = env_ids.detach().cpu().numpy()
    a = np.asarray(env_ids)
    if a.ndim != 1 or a.size == 0 or not np.issubdtype(a.dtype, np.integer):
        raise ValueError("env_ids must be a non-empty 1-D sequence of integers")
    if int(a.min()) < 0 or int(a.max()) >= num_envs:
        raise ValueError(f"env_ids must lie in [0, {num_envs})")
    return np.ascontiguousarray(a, dtype=np.int32)


def check_channels(channels: int) -> int:
    if channels not in (1, 3):
        raise ValueError("channels must be 1 (grey) or 3 (RGB)")
    return int(channels)


def decode_target(torch, out, n: int, channels: int, device):
    """`out` for n decoded frames: a new uint8 [n, 144, 160, channels] tensor, or the caller's, checked."""
    shape = (n, *FRAME_SHAPE, channels)
    if out is None:
        return torch.empty(shape, dtype=torch.uint8, device=device)
    ok = (torch.is_tensor(out) and out.dtype == torch.uint8 and out.device == device and out.is_contiguous() and tuple(out.shape) == shape
          and out.data_ptr() % 16 == 0)
    if not ok:  # the kernel writes n * 23,040 * channels bytes at out's address in 16-byte stores
        raise ValueError(f"out must be a contiguous, 16-byte aligned uint8 tensor {list(shape)} on {device}")
    return out


class FrameRecorder:
    """The frame of every step of the envs `env_ids`, in a device ring of `capacity` steps, with the same steps' done flags.

    Created by VecEnvironment.record_frames.  Each VecEnvironment.step queues one capture after the step's kernels and before
    its auto-reset, so the last frame of an episode that just ended is recorded, not the frame after the reset; an env that
    sits a step out (`skip`) records its unchanged frame.  The slot counter lives on the host: recording never waits for the
    device.  When more steps than `capacity` have been recorded, the oldest are overwritten.
    """

    def __init__(self, vec, env_ids, capacity: int):
        torch = vec.torch
        if int(capacity) < 1:
            raise ValueError("capacity must be at least 1")
        self.vec = vec
        self.capacity = int(capacity)
        self.env_ids = host_env_ids(env_ids, vec.num_envs)
        n = self.env_ids.size
        with torch.cuda.device(vec.device):
            self._ids = torch.from_numpy(self.env_ids).to(vec.device)
            self._ids_long = self._ids.long()
            self._ring = torch.empty((self.capacity, n, _capi.FRAME_WORDS), dtype=torch.int32, device=vec.device)  # uint32 words
            self._done = torch.zeros((self.capacity, n), dtype=torch.bool, device=vec.device)
        self._recorded = 0  # captures since creation or clear()

    def _capture(self, done, stream: int):
        """One step's frames and done flags into the next slot (VecEnvironment.step calls this)."""
        slot = self._recorded % self.capacity
        self.vec.handle.capture_frames(self._ring[slot], self._ids, stream=stream)
        self._done[slot] = done[self._ids_long].bool()
        self._recorded += 1

    @property
    def count(self) -> int:
        """Steps held: the number recorded, up to capacity."""
        return min(self._recorded, self.capacity)

    def _segments(self, start: int = 0, stop=None):
        """Ring slots of the chronological steps [start, stop) as at most two contiguous ranges (the ring wraps once)."""
        lo, hi, _ = slice(start, stop).indices(self.count)
        head = self._recorded % self.capacity if self._recorded > self.capacity else 0  # slot of the oldest step held
        segs = []
        while lo < hi:
            s = (head + lo) % self.capacity
            k = min(hi - lo, self.capacity - s)
            segs.append((s, s + k))
            lo += k
        return segs

    def packed(self):
        """uint32 [count, n, FRAME_WORDS] device tensor: the packed frames, oldest step first.  Until the ring wraps this is a
        view of the ring, which later steps overwrite; after that, a copy."""
        torch = self.vec.torch
        segs = self._segments()
        if len(segs) == 1:
            return self._ring[segs[0][0]:segs[0][1]].view(torch.uint32)
        parts = [self._ring[a:b] for a, b in segs]
        return (torch.cat(parts) if parts else self._ring[:0]).view(torch.uint32)

    def frames(self, channels: int = 3, start: int = 0, stop=None):
        """uint8 [steps, n, 144, 160, channels] device tensor of the recorded steps [start, stop) in chronological order
        (Python slice bounds over the `count` steps held), decoded on the device: channels 1 = grey, 3 = RGB as screen()."""
        torch = self.vec.torch
        channels = check_channels(channels)
        segs = self._segments(start, stop)
        n = self.env_ids.size
        steps = sum(b - a for a, b in segs)
        out = torch.empty((steps, n, *FRAME_SHAPE, channels), dtype=torch.uint8, device=self.vec.device)
        k = 0
        for a, b in segs:
            self.vec.handle.frames_to_rgb(self._ring[a:b].view(-1, _capi.FRAME_WORDS), out[k:k + b - a], channels, stream=self.vec._stream())
            k += b - a
        return out

    def dones(self):
        """bool [count, n] device tensor: the done flag each recorded step returned for each env, oldest step first."""
        torch = self.vec.torch
        parts = [self._done[a:b] for a, b in self._segments()]
        return torch.cat(parts) if len(parts) > 1 else (parts[0] if parts else self._done[:0])

    def clear(self):
        """Empties the ring; recording goes on from the next step."""
        self._recorded = 0
