"""B200-native ensemble-HMC engine behind the Python surface of
Anton-Le/PhysicsBasedBayesianInference (``Ensemble``, ``Leapfrog`` / ``StormerVerlet``,
``HMC.getSamples``, ``potential``).

Host code is Python; all arithmetic of the hot path runs in hand-written sm_100a
CUDA kernels reached through the ctypes C-ABI declared in ``include/ehmc.h``
(``_ehmc.so``, built in-tree by ``build.build_library``).  There is no CPU
fallback: without the library or without a CUDA device every compute call raises.

For scripts written against the reference's flat modules
(``from ensemble import Ensemble``), put ``physicsbasedbayesianinference_b200/flat``
on ``sys.path``.
"""
from . import _lib  # noqa: F401
from .ensemble import Ensemble, boltzmannConst  # noqa: F401
from .integrator import Integrator, Leapfrog, StormerVerlet  # noqa: F401
from .HMC import HMC, GaussianDensity  # noqa: F401
from . import potential  # noqa: F401
from . import diagnostics, io, numpyro_adapter, parallel  # noqa: F401
from .potential import (  # noqa: F401
    CoinTossPotential,
    FunnelPotential,
    GaussianPotential,
    HarmonicPotential,
    HierarchicalNormalPotential,
    LogisticPotential,
    NBodyPotential,
    Potential,
    harmonicPotentialND,
)

__version__ = "0.1.0"
