"""voldor_b200 — B200-native (sm_100a) implementation of VOLDOR's per-window EM inference hot path.

The compute lives in voldor_b200/libvoldor_b200.so (hand-written CUDA, built in-tree by `make lib` or
`__graft_entry__.build()`).  There is no CPU fallback: importing the bindings without the library, or
calling them without a CUDA device, raises."""
import os as _os

# hardware work queues for several windows in flight (see csrc/context.cu); only effective before CUDA is initialised
_os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

from .pyvoldor_vo import (voldor, load_library, set_bootstrap_override, voldor_ex, select_context,  # noqa: F401
                          context_srand, set_device)
from .falign import falign, falign_ex  # noqa: F401,E402

__all__ = ["voldor", "voldor_ex", "falign", "falign_ex", "load_library", "set_bootstrap_override", "select_context",
           "context_srand", "set_device"]
