"""pyfocusr_b200 -- B200-native (sm_100a) drop-in for the spectral-correspondence hot path of
gattia/pyfocusr.  ``import pyfocusr_b200 as pyfocusr`` gives the reference's names:
``Focusr``, ``Graph``, ``recursive_eig``, ``eigsort`` (reference pyfocusr/__init__.py:1-5), plus
``PolyData`` / ``read_vtk_mesh`` for VTK-free mesh IO and ``SpectralBatch`` for batched pairs.

All arithmetic of the hot path runs in ``csrc/libfocusr_b200.so`` (hand-written CUDA behind the C
ABI of include/focusr_b200.h); there is no CPU fallback.
"""
from . import mesh as vtk_functions  # read_vtk_mesh lives here (reference: vtk_functions.py:5-9)
from .batch import SpectralBatch
from .eigsort import eigsort
from .focusr import Focusr
from .graph import Graph, recursive_eig
from .mesh import PolyData, ellipsoid_pair, icosphere, perturbed_ellipsoid, read_vtk_mesh, write_vtk_mesh
from .surface import surface_distances

__all__ = [
    "Focusr", "Graph", "recursive_eig", "eigsort", "SpectralBatch", "PolyData", "read_vtk_mesh", "write_vtk_mesh",
    "icosphere", "perturbed_ellipsoid", "ellipsoid_pair", "vtk_functions", "surface_distances",
]
__version__ = "0.1.0"
