"""Drop-in mirror of `pytorch3d.pathtracer` for the per-ray hot path (SURVEY.md section 8b):
same class names, constructor arguments, attributes and method signatures; the bodies call the
fused CUDA kernels of libnrt_b200."""
from .interaction import DirectionSample, Interaction, MixedInteraction, SurfaceInteraction
from .integrators import Debug, Direct, Mask, NeRFIntegrator, NeRFReproduce, Path, Silhouette
from .samplers import Sampler
from .main import pathtrace, pathtrace_sample
from .utils import LossSampler
from .neural_blocks import SkipConnMLP
from . import bsdf, cameras, checkpoint, integrators, lights, mesh, shapes, training_utils, utils, warps  # noqa: F401

__all__ = [k for k in globals().keys() if not k.startswith("_")]
