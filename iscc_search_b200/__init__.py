"""
iscc_search_b200 - B200-native exact NPHD / Hamming top-k backend for iscc-search.

Public surface:
    B200IndexManager, B200Index        IsccIndexProtocol backend (drop-in for iscc-search's usearch:/// backend)
    ShardedNphdIndex, ShardedIndex128, Matches, BatchMatches, timer
                                       what iscc-search imports from `iscc_usearch` (vector-store boundary)
All search arithmetic runs in libisx_b200.so (hand-written sm_100a CUDA); there is no CPU path.
"""

from iscc_search_b200.matches import BatchMatches, JoinPairs, Match, Matches  # noqa: F401
from iscc_search_b200.nphd import MultiDeviceIndex128, MultiDeviceNphdIndex, ShardedIndex128, ShardedNphdIndex  # noqa: F401
from iscc_search_b200.utils import timer  # noqa: F401
from iscc_search_b200.backend import B200Index, B200IndexManager  # noqa: F401

__all__ = ["B200IndexManager", "B200Index", "ShardedNphdIndex", "MultiDeviceNphdIndex", "ShardedIndex128", "MultiDeviceIndex128", "Matches", "BatchMatches", "Match", "JoinPairs", "timer"]
__version__ = "0.1.0"
