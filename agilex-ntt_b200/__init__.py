"""agilex-ntt_b200: B200-native (sm_100a) drop-in for the hot path of joekurina/Agilex-NTT -- the negacyclic
forward / inverse NTT over 30-bit-class primes and the NTT-based negacyclic polynomial multiply.

Layout: csrc/ (CUDA kernels + the C ABI of include/agxntt.h), host/ (C++ mirror of the reference's kernel API and
a main.cpp-shaped driver), binding.py (ctypes over the C ABI), sharding.py (multi-GPU batch partition).
The directory name carries a hyphen, so import it as `agilex_ntt_b200` (root-level alias module).
"""
from .binding import AgxError, Context, Context64, RefPipeline, EXPORTS, error_string, galois_element, lib  # noqa: F401
from .sharding import shard_bounds, all_shards, combine_checksums  # noqa: F401
from . import build  # noqa: F401
