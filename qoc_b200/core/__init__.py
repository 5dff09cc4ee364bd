"""
core - the programs of the qoc API (mirror of qoc.core).
"""
from .lindbladdiscrete import evolve_lindblad_discrete, grape_lindblad_discrete, grape_lindblad_discrete_batch
from .schroedingerdiscrete import (evolve_schroedinger_discrete, evaluate_schroedinger_discrete,
                                   grape_schroedinger_discrete, grape_schroedinger_discrete_batch)

__all__ = ["evolve_lindblad_discrete", "grape_lindblad_discrete", "grape_lindblad_discrete_batch", "evolve_schroedinger_discrete",
           "evaluate_schroedinger_discrete", "grape_schroedinger_discrete",
           "grape_schroedinger_discrete_batch"]
