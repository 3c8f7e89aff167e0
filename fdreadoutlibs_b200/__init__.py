"""fdreadoutlibs_b200 — B200-native software trigger-primitive generation behind the fdreadoutlibs frame-processor path.

Only the hot path lives here (DESIGN.md): CUDA kernels + C ABI (`csrc/`, `include/swtpg.h`), this thin ctypes face, and the
host C++ mirror of the reference's FrameProcessor interface (`host/`). Importing the package loads libswtpg_b200.so and
fails loudly if it has not been built.
"""
from . import frames  # noqa: F401
from .api import (ALGORITHMS, PinnedBuffer, SwtpgError, TPGAlgorithmInexistent, TPGenerator, channel_covariance, device_available,  # noqa: F401
                  firwin_int, gen_params, gen_wib2_device, gen_wib2_host, gen_wibeth_device, gen_wibeth_host, merge_sorted, noise_frequencies, noise_power, sort_tps)

__all__ = ["frames", "TPGenerator", "PinnedBuffer", "SwtpgError", "TPGAlgorithmInexistent", "ALGORITHMS", "channel_covariance", "device_available", "firwin_int",
           "gen_params", "gen_wibeth_host", "gen_wib2_host", "gen_wibeth_device", "gen_wib2_device", "merge_sorted", "noise_frequencies",
           "noise_power", "sort_tps"]
