"""pokegym_b200 -- B200-native batched Game Boy environment, drop-in for pokegym's Environment.

Only the hot path of the reference (`Environment.reset/step` over PyBoy) is implemented, as
hand-written CUDA for sm_100a behind the C ABI of include/gbenv.h.  Importing this package does not
load the CUDA library; constructing an environment does, and fails loudly when it is missing.
"""
from .version import __version__  # noqa: F401


def __getattr__(name):
    if name in ("Environment", "VecEnvironment", "Box", "Discrete"):
        from . import vec_env

        return getattr(vec_env, name)
    if name == "FrameRecorder":
        from . import frames

        return frames.FrameRecorder
    if name == "EnvGroups":
        from . import groups

        return groups.EnvGroups
    raise AttributeError(name)
