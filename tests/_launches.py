"""CUPTI launch counts of this library's kernels (csrc/launch_count.cu), for tests that prove which kernel route a call
takes."""
import ctypes

import torch


def count_launches(fn):
    """-> {kernel (mangled name): launches} of this library during fn(), or None when CUPTI cannot be used."""
    from pytorch_speaker_verification_b200 import _lib
    L = _lib.lib()
    if L.svb_launch_count_begin() != 0:
        return None
    try:
        fn()
        torch.cuda.synchronize()
    finally:
        ours, other = ctypes.c_longlong(0), ctypes.c_longlong(0)
        names = ctypes.create_string_buffer(1 << 16)
        L.svb_launch_count_end(ctypes.byref(ours), ctypes.byref(other), names, ctypes.c_size_t(len(names)))
    per = {}
    for item in names.value.decode().split(";"):
        if "=" in item:
            k, n = item.rsplit("=", 1)
            per[k] = int(n)
    return per


def launched(names, *parts):
    """True when some launched kernel's mangled name contains every one of ``parts``."""
    return any(all(p in k for p in parts) for k in names)
