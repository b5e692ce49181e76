"""grakel_b200 -- B200-native graph-kernel Gram engine behind the GraKeL operator API.

Hot path only: WeisfeilerLehman (subtree, or over EdgeHistogram / ShortestPath), VertexHistogram,
EdgeHistogram, ShortestPath, ShortestPathAttr, WeisfeilerLehmanOptimalAssignment, NeighborhoodHash, CoreFramework (`fit` / `transform` /
`fit_transform` / `diagonal`), plus the `GraphKernel` name dispatcher.  All kernel matrices are computed by hand-written sm_100a CUDA
(`libgrakel_b200.so`, C-ABI in include/grakel_b200.h); there is no CPU path.
"""
from .packing import Graph
from .kernels import (EdgeHistogram, Kernel, NeighborhoodHash, ShortestPath, ShortestPathAttr, VertexHistogram,
                      WeisfeilerLehman, WeisfeilerLehmanOptimalAssignment)
from .core_framework import CoreFramework
from .graph_kernels import GraphKernel
from ._lib import default_device, set_default_device

__version__ = "0.1.0"
__all__ = ["Graph", "Kernel", "GraphKernel", "WeisfeilerLehman", "VertexHistogram", "ShortestPath",
           "ShortestPathAttr", "EdgeHistogram", "CoreFramework", "WeisfeilerLehmanOptimalAssignment", "NeighborhoodHash",
           "set_default_device",
           "default_device"]
