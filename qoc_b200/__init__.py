"""
qoc_b200 - B200-native (sm_100a) implementation of the GRAPE propagate-and-differentiate hot path of
SchusterLab/qoc behind qoc's own Python API.  `import qoc_b200 as qoc` is the drop-in.
"""
from .core import (evolve_lindblad_discrete, evolve_schroedinger_discrete, evaluate_schroedinger_discrete,
                   grape_lindblad_discrete, grape_lindblad_discrete_batch, grape_schroedinger_discrete,
                   grape_schroedinger_discrete_batch)

__all__ = ["evolve_lindblad_discrete", "evolve_schroedinger_discrete", "evaluate_schroedinger_discrete",
           "grape_lindblad_discrete", "grape_lindblad_discrete_batch", "grape_schroedinger_discrete",
           "grape_schroedinger_discrete_batch"]
