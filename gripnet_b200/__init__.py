"""gripnet_b200 — B200-native GripNet supergraph message passing.

Drop-in for the reference ``gripnet`` package's hot path:

    import gripnet_b200
    gripnet_b200.install_as_gripnet()          # `from gripnet.layers import homoGraph` now resolves here
    from gripnet.layers import homoGraph, interGraph
    from gripnet.decoder import multiRelaInnerProductDecoder

Host code is Python/PyTorch (device memory, streams, autograd); all arithmetic is
hand-written CUDA for sm_100a behind the C ABI of ``include/gripnet_b200.h``.
There is no CPU fallback.
"""
import sys

from . import _lib
from ._lib import GripnetLibraryError, launch_count  # noqa: F401

__version__ = "0.1.0"


def _require_library():
    _lib.load()


_require_library()          # fail loudly at import if libgripnet_b200.so is missing

from . import graph, ops, parallel, layers, decoder, encoder, losses, utils, metrics, optim, ranking  # noqa: E402,F401
from .layers import myGCN, myRGCN, homoGraph, interGraph  # noqa: E402,F401
from .decoder import multiRelaInnerProductDecoder, multiClassInnerProductDecoder  # noqa: E402,F401
from .losses import link_prediction_loss, node_classification_loss  # noqa: E402,F401
from .ranking import EdgeFilter, LinkRanker, PairRanker, RelationRanker  # noqa: E402,F401


def install_as_gripnet():
    """Register this package under the reference's import name ``gripnet``."""
    me = sys.modules[__name__]
    sys.modules["gripnet"] = me
    for name in ("layers", "decoder", "encoder", "utils"):
        sys.modules["gripnet." + name] = getattr(me, name)
    return me
