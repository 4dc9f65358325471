"""B200-native SLOD offline phase: CUDA library (csrc/ -> libslod_b200.so) + ctypes binding.

The directory name carries a hyphen (it mirrors the reference repo name); import it with
``importlib.import_module("dealii-slod_b200")`` or through the alias module ``slod_b200`` at the repo root.
"""
from .binding import (EXPORTS, LIB_PATH, PLAN_KEYS, PROBLEM_DIFFUSION, PROBLEM_ELASTICITY, SlodContext,  # noqa: F401
                      SlodError, SlodParams, load_library)
from .build import build_library  # noqa: F401
