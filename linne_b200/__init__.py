"""linne_b200 -- B200-native (sm_100a) implementation of the LINNE lossless codec's block
encode/decode path, behind the reference's own C API.

    from linne_b200 import Product
    codec = Product()                      # loads liblinne_b200.so; raises if it is not built
    stream = codec.encode(pcm_int32_planar, bits=16, preset=7)
    pcm = codec.decode(stream)

Everything heavy lives in linne_b200/csrc (host C + CUDA); this package is a thin ctypes mirror.
"""
from .api import (Product, LinneApi, load_library, EncoderSession, DecoderSession, DeviceBuffer, PeerMapping, ChannelParams, FileDesc, SeekPoint, Window, LINNEHeader, LINNEEncodeParameter,  # noqa: F401
                  LINNEEncoderConfig, LINNEDecoderConfig, OK, INVALID_ARGUMENT, INVALID_FORMAT,
                  INSUFFICIENT_BUFFER, INSUFFICIENT_DATA, PARAMETER_NOT_SET, DATA_CORRUPTION, NG)
