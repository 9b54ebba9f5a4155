"""liorf_b200 — B200-native (sm_100a) scan-to-map registration hot path of liorf behind a C ABI.

The package holds only what the path needs: `csrc/` (CUDA kernels + the C ABI, built into `lib/libliorf_b200.so`),
`host/` (C++ mirror of the reference's member-function interface) and this thin ctypes binding used by the tests
and the benchmark.  There is no CPU fallback: importing works without a GPU (so the build can be checked), but every
compute call needs the CUDA library and a device.
"""
import os as _os

# one hardware channel per stream (read by the CUDA driver at context creation; harmless if CUDA is already up): see DESIGN.md §7
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from ._lib import load_library, library_path, build_library  # noqa: F401,E402
from .api import imuDeskewInfo, sc_tree_schedule, Context, Params, LMTrace, FrameIn, FrameOut, CloudInfoGuess, GuessState, P4, PRAW  # noqa: F401
