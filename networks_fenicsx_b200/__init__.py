"""B200-native hydraulic-network assemble-and-solve path behind the ``networks_fenicsx`` API.

Intended switch in a user script::

    import networks_fenicsx_b200 as networks_fenicsx

The three classes and two helper modules the reference exports are available under the same names
(``HydraulicNetworkAssembler``, ``NetworkMesh``, ``Solver``, ``network_generation``,
``post_processing``); ``fem`` / ``la`` hold the DOLFINx / PETSc stand-ins the calls return,
``distributed`` / ``parallel`` the multi-GPU layer (``PartitionedSolver``: one network cut over several
GPUs, or into several parts on one GPU, from a single process), ``common`` the timer registry.
"""

from . import common, fem, la, network_generation, post_processing  # noqa: F401
from .assembly import HydraulicNetworkAssembler
from .distributed import PartitionedSolver
from .mesh import NetworkMesh
from .solver import Solver

__version__ = "0.1.0"
__program_name__ = "networks_fenicsx_b200"
__license__ = "MIT"
__author__ = ""
__email__ = ""

__all__ = sorted(
    ["NetworkMesh", "HydraulicNetworkAssembler", "Solver", "PartitionedSolver", "network_generation",
     "post_processing", "fem", "la", "common"]
)
