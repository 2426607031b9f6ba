"""optable_b200: a B200-native ray-propagation engine behind optable's Python API.

`from optable_b200 import *` gives the names user scripts take from `from optable import *`: Ray, the leaf
components, the assemblies, Monitor, OpticalTable, the materials. The bounce loop runs in liboptb.so
(hand-written sm_100a CUDA behind the C ABI of include/optb.h); there is no CPU fallback.
"""
from .pose import Base, Vector
from .materials import (Material, ConstMaterial, Vacuum, SellmeierMaterial, RefractiveIndex, Glass_NBK7, Glass_UVFS,
                        Glass_NSF5, Glass_NSF11, Glass_NSK2, Glass_NSF57)
from .shapes import Surface, Point, Plane, Circle, Rectangle, Cylinder, Sphere, ASphere, Polygon
from .rays import GaussianBeam, Ray, multiplex_rays_in_wavelength
from .elements import (OpticalComponent, PointObj, Block, BaseMirror, BaseRefraciveSurface, Mirror, SquareMirror,
                       SquareRefractive, CircleRefractive, SphereRefractive, BeamSplitter, Lens, CylMirror)
from .assemblies import (ComponentGroup, GlassSlab, CircleGlassSlab, MLA, MMA, MMADisordered, DMD, WedgePlate,
                         MirrorPair, Prism, TriangularPrism, MirrorPrism, MirrorCube, DovePrism, PlanoConvexLens,
                         BiConvexLens, Doublet, ASphericLens, ASphericExactSphericalLens, ASphericParametricLens)
from .monitors import Monitor
from .solvers import solve_ray_bboxes_intersections, solve_ray_ray_intersection, solve_normal_to_normal_rotation
from .table import OpticalTable, install, trace_table
from .sweep import SweepABCD, SweepResult, SweepScene, sweep_abcd_matrix, trace_sweep

__all__ = [n for n in dir() if not n.startswith("_")]
