"""loc_lib_b200 — B200-native scan-to-map registration (ICP P2P / P2Line / P2Plane, direct and incremental NDT, LOAM).

One hot path of maotian123/loc_lib rebuilt for sm_100a behind the reference's MatchingInterface:
see DESIGN.md for the scope and INTEGRATION.md for the drop-in binding.
"""
from .registration import (IcpMethod, IcpOptions, IcpRegistration, NdtMethod, NdtNearbyType, NdtOptions,  # noqa: F401
                           NdtRegistration, LoamRegistration, LocTracker, LioTracker, se3_inv, se3_mul)
from ._lib import LOOP_GRAPH, LOOP_PERSISTENT  # noqa: F401
