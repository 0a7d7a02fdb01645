"""b200-blockdct: B200-native 8x8 block DCT -> quantise -> IDCT (drop-in for the hot path
of GerryDps/CUDA-DCT-IDCT).

The product is the CUDA library built from ``csrc/`` (``libb200dct.so``: the C ABI of
``include/b200dct.h``; ``libb200dct_compat.so``: the reference's own C++ entry points).
This package is only the thin Python host side over that C ABI: ctypes bindings that
take torch CUDA tensors (device memory, streams) or numpy host arrays.  There is no
CPU fallback -- importing works anywhere, computing requires the built library and a GPU.
"""
from .api import (  # noqa: F401
    ALL_COEFFS,
    B200DCTError,
    HostPipeline,
    Plan,
    dct_all_blocks,
    dct_all_blocks_cuda,
    forward,
    idct_all_blocks,
    idct_all_blocks_cuda,
    inverse,
    lib,
    lib_path,
    metrics,
    roundtrip,
    roundtrip_any,
    roundtrip_batch,
    ImageBatch,
    roundtrip_host,
    roundtrip_rgb,
    forward_rgb,
    inverse_rgb,
    coded_bits,
    compression_factor,
    roundtrip_with_metrics,
    zigzag_mask,
)
from . import api, dist, imageio  # noqa: F401
from .build import build  # noqa: F401
from .stripes import batch_images, stripe_rows  # noqa: F401

__all__ = [
    "ALL_COEFFS", "B200DCTError", "HostPipeline", "Plan", "build", "dct_all_blocks", "dct_all_blocks_cuda", "forward",
    "idct_all_blocks", "idct_all_blocks_cuda", "inverse", "lib", "lib_path", "metrics", "roundtrip",
    "roundtrip_any", "roundtrip_batch", "ImageBatch", "roundtrip_host", "roundtrip_rgb", "forward_rgb", "inverse_rgb", "coded_bits", "compression_factor", "roundtrip_with_metrics", "stripe_rows", "batch_images", "zigzag_mask",
]
