"""dot_ring_b200: B200-native (sm_100a) ring-proof engine behind dot-ring's Python API.

Host code is Python and calls the CUDA library ``libdotring_b200.so`` through ctypes
(``dot_ring_b200._native``).  The library is loaded on first use and its absence is a hard
``ImportError``: there is no CPU fallback.

Public names mirror ``dot_ring`` (dot_ring/__init__.py:32-77) for the path this engine covers.
"""

from .curve import Bandersnatch, Bandersnatch_SHAKE128
from .kzg import KZG
from .params import RingProofParams
from .ring import Ring, RingRoot, RingVerifier
from .ring_proof import RingProof
from .vrf import PedersenVRF, RingVRF, ThinVRF, TinyVRF

__all__ = ["Bandersnatch", "Bandersnatch_SHAKE128", "KZG", "RingProofParams", "Ring", "RingRoot", "RingVerifier", "RingProof", "RingVRF", "PedersenVRF", "TinyVRF", "ThinVRF", "__version__"]
__version__ = "0.1.0"
