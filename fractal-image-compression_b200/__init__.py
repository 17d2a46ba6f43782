"""fractal-image-compression_b200: B200-native (sm_100a) drop-in for the encode/decode hot
path of LariWa/Fractal-Image-Compression.  The product is the C-ABI library
lib/libfic_b200.so (include/fic_b200.h); this package is its host-side mirror of the
reference's codec interface plus the torch.distributed plumbing for multi-GPU encodes.
"""
from . import _lib, synth
from ._lib import (FIC_ENGINE_AUTO, FIC_ENGINE_DIRECT, FIC_ENGINE_FUSED, FIC_ENGINE_UMMA, FIC_UMMA_KIND_AUTO, FIC_UMMA_KIND_F16,
                   FIC_UMMA_KIND_I8, FIC_UMMA_PAIR_AUTO, FIC_UMMA_PAIR_OFF, FIC_UMMA_PAIR_ON, FIC_MODE_GREY, FIC_MODE_RGB, FIC_MODE_GREY_ISO, FIC_MODE_GREY_QT, FIC_MODE_RGB_QT, ABI_SYMBOLS, LIB_PATH, FicError, Timings)
from .codec import ByteSink, FractalCompression, Handle, MultiHandle, RasterImage, quadtree_stream_info, stream_read, stream_write

__all__ = [
    "ABI_SYMBOLS", "ByteSink", "FIC_ENGINE_AUTO", "FIC_ENGINE_DIRECT", "FIC_ENGINE_FUSED", "FIC_ENGINE_UMMA", "FIC_MODE_GREY", "FIC_MODE_GREY_ISO",
    "FIC_MODE_GREY_QT", "FIC_MODE_RGB", "FIC_MODE_RGB_QT", "FIC_UMMA_KIND_AUTO",
    "FIC_UMMA_KIND_F16", "FIC_UMMA_KIND_I8", "FIC_UMMA_PAIR_AUTO", "FIC_UMMA_PAIR_OFF", "FIC_UMMA_PAIR_ON", "FicError",
    "FractalCompression", "Handle", "LIB_PATH", "MultiHandle", "RasterImage", "Timings", "quadtree_stream_info", "stream_read", "stream_write", "synth",
]
