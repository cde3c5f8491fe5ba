"""PufferLib-shaped vector adaptor (SURVEY.md section 8f-1): async_reset / recv / send over VecEnvironment.

The reference is driven by a PufferLib fork (README.md:40, :116-118) that is neither in the reference tree nor installed
here, so the contract is restated from PufferLib's published vector API (pufferlib.vector Serial / Multiprocessing, 1.0):

  * observations are flat uint8 [N, 23040] (the emulation layer flattens the (72, 80, 4) Box), or [N, 2304] over a
    VecEnvironment with obs_format="packed" (the trainer decodes minibatches with VecEnvironment.unpack_obs);
  * `recv()` returns (obs, rewards, terminals, truncations, infos, env_ids, mask);
  * an env that reported `done` is reset on the NEXT `send`: that call's action for it is ignored, it is not stepped, and
    `recv` delivers its reset observation with reward 0 and terminal False (pufferlib.vector.Serial.send: `if env.done:
    o, i = env.reset() ... else: o, r, d, t, i = env.step(atn)`);
  * infos: one dict per env that finished an episode on this step.  By default that is the env's stats and reward terms
    (info_row_to_dict); with full_infos=True it is the reference's whole info dict (VecEnvironment.episode_infos: the
    130 event flags and the detailed rewards too), without the per-env exploration map.

Everything stays on the device: the reset is masked by the previous step's done vector (gbenv_reset_dev) and the same vector
makes those envs sit the step out (gbenv_step_masked); only the per-episode info rows of finished envs come to the host.
"""
from __future__ import annotations

import numpy as np

from .info import info_row_to_dict
from .vec_env import VecEnvironment


class PufferVecAdaptor:
    def __init__(self, vec: VecEnvironment, full_infos: bool = False):
        if vec.auto_reset:
            raise ValueError("PufferVecAdaptor does the resets itself: construct the VecEnvironment with auto_reset=False")
        self.vec = vec
        self.full_infos = bool(full_infos)
        self.num_envs = vec.num_envs
        self.env_ids = np.arange(self.num_envs)
        self._row_bytes = int(np.prod(vec.observation_space.shape))
        t = vec.torch
        self._pending = t.zeros(self.num_envs, dtype=t.uint8, device=vec.device)  # envs whose episode ended on the last step
        self._any_pending = False
        self._last = None

    def async_reset(self, seed=None):
        obs, _ = self.vec.reset()
        t = self.vec.torch
        self._pending.zero_()
        self._any_pending = False
        self._last = (obs, t.zeros(self.num_envs, dtype=t.float64, device=self.vec.device), t.zeros(self.num_envs, dtype=t.bool, device=self.vec.device), [])

    def send(self, actions):
        if self._any_pending:  # reset instead of step for the envs that finished; their action is ignored
            self.vec.reset(mask=self._pending)
            obs, rew, done, _, _ = self.vec.step(actions, skip=self._pending)
        else:
            obs, rew, done, _, _ = self.vec.step(actions)
        infos = []
        self._pending.copy_(done)
        self._any_pending = bool(done.any())  # the one host read per step; PufferLib inspects the dones on the host anyway
        if self._any_pending and self.full_infos:
            infos = list(self.vec.episode_infos(done).values())
        elif self._any_pending:
            rows = self.vec.info().cpu().numpy()
            infos = [info_row_to_dict(rows[e]) for e in np.nonzero(done.cpu().numpy())[0]]
        self._last = (obs, rew, done, infos)

    def recv(self):
        obs, rew, done, infos = self._last
        flat = obs.reshape(self.num_envs, self._row_bytes)
        mask = np.ones(self.num_envs, dtype=bool)
        return flat, rew, done, done, infos, self.env_ids, mask
