"""smokephysai_b200 -- B200-native (sm_100a) implementation of SmokePhysAI's grid smoke-simulation step.

Scope: the hot path of the reference's src/physics (NavierStokesSimulator.step and its SmokeSimulator
facade) behind the reference's own Python class surface.  Kernels live in csrc/*.cu, exposed through the
C ABI in include/smoke_b200.h (libsmoke_sm100.so); there is no CPU or eager-PyTorch fallback.
"""
from .navier_stokes import NavierStokesSimulator, FieldLayout  # noqa: F401
from .fractal_generator import FractalGenerator  # noqa: F401
from .smoke_simulator import SmokeSimulator  # noqa: F401
from . import autodiff  # noqa: F401

__all__ = ["NavierStokesSimulator", "FractalGenerator", "SmokeSimulator", "FieldLayout", "autodiff"]
