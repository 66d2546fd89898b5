"""neumesh_b200 - B200-native implementation of the NeuMesh volumetric-rendering hot path.

Public surface (mirrors the reference's Python API for this path):

* ``NeuMesh``           <- models/frameworks/neumesh/neumesh.py
* ``MeshGrid``          <- models/mesh_grid.py
* ``frnn_grid_points``  <- third-party ``frnn`` (models/mesh_grid.py:64,109)
* ``volume_render`` / ``SingleRenderer`` <- models/renderer.py
* ``TextureEditableNeuMesh`` <- editing/texture_neumesh/texture_neumesh.py
* ``extract_mesh`` / ``marching_cubes`` <- extract_mesh.py / third-party ``mcubes.marching_cubes``
* ``parallel.render_sharded`` <- the ``nn.DataParallel`` ray scatter / gather of models/trainer.py:39-42

The compute lives in ``lib/libneumesh_b200.so`` (hand-written sm_100a CUDA behind the C ABI of
``include/neumesh_b200.h``); importing this package does not load it, using it does - and fails loudly if the
extension is missing: there is no CPU fallback.
"""
from .mesh_grid import GridHandle, MeshGrid, MeshPrimitive, frnn_grid_points  # noqa: F401
from .neumesh import Embedder, NeuMesh, get_embedder, interpolation  # noqa: F401
from .renderer import SingleRenderer, release_workspace, volume_render  # noqa: F401
from .texture_neumesh import TextureEditableNeuMesh  # noqa: F401
from .neus import NeuS  # noqa: F401
from .mesh_extraction import extract_mesh, marching_cubes  # noqa: F401
from . import parallel  # noqa: F401

__all__ = ["NeuMesh", "MeshGrid", "MeshPrimitive", "GridHandle", "frnn_grid_points", "volume_render",
           "release_workspace", "TextureEditableNeuMesh", "SingleRenderer", "Embedder", "get_embedder",
           "interpolation", "parallel", "NeuS", "extract_mesh", "marching_cubes"]
