"""mfmarl_b200 -- batched, device-resident face of the B200 battle / Ising kernels.

Thin ctypes layer over build/libmagent.so (C ABI: include/mfmarl_batched.h).  PyTorch tensors are the
buffers (device memory, streams); the engine never runs on the CPU.
"""
from .lib import load_library, LIB_PATH
from .battle import BatchedGridWorld, decode_env_state, mean_action
from .ising import IsingMFQ, IsingMetropolis, IsingSwendsenWang

__all__ = ["load_library", "LIB_PATH", "BatchedGridWorld", "decode_env_state", "mean_action", "IsingMFQ", "IsingMetropolis",
           "IsingSwendsenWang"]
