"""stag_b200 -- B200-native stochastic neighbour aggregation, drop-in for the hot path of
yuanqing-wang/stag (``stag.layers`` / ``stag.models`` / ``stag.zoo`` / ``stag.distributions``
/ ``stag.likelihoods`` keep their constructors, forward signatures and state_dict keys).

Everything below the Python modules runs in ``_C/libstag_b200.so`` (hand-written sm_100a
CUDA behind the C ABI of ``include/stag_b200.h``).  There is no CPU fallback: operators
raise ``StagLibraryError`` when the library is missing or a tensor is not on a CUDA device.
"""
from . import _lib, random  # noqa: F401
from . import distributions, likelihoods, utils, graph, function, ops, calibration  # noqa: F401
from . import layers, models, zoo  # noqa: F401
from .graph import (Graph, as_graph, batch, rand_graph, add_self_loop, remove_self_loop,  # noqa: F401
                    add_reverse_edges, sum_nodes, mean_nodes)
from .random import manual_seed  # noqa: F401
from ._lib import StagLibraryError, StagError  # noqa: F401

__version__ = "0.1.0"
