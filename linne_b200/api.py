"""linne_b200.api -- ctypes mirror of the LINNE C API as served by liblinne_b200.so.

The public structs and the 14 entry points keep the reference's names, argument meaning and
result codes (include/linne.h, linne_encoder.h, linne_decoder.h).  `LinneApi` drives any
library that exports that API; `load_library()` loads the CUDA product and fails loudly if it
has not been built -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import numpy as np

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
PRODUCT_SO = os.path.join(PKG_DIR, "liblinne_b200.so")

OK, INVALID_ARGUMENT, INVALID_FORMAT, INSUFFICIENT_BUFFER, INSUFFICIENT_DATA, \
    PARAMETER_NOT_SET, DATA_CORRUPTION, NG = range(8)

PRESET_LAYERS = {0: (2, 32), 1: (2, 32), 2: (4, 64, 8), 3: (4, 64, 8), 4: (4, 64, 8),
                 5: (4, 128, 16), 6: (4, 128, 16), 7: (4, 128, 16)}


# ----------------------------------------------------------------------------------------------
# ctypes mirrors of the public structs (include/linne.h, linne_encoder.h, linne_decoder.h)
# ----------------------------------------------------------------------------------------------
class LINNEHeader(C.Structure):
    _fields_ = [("format_version", C.c_uint32), ("codec_version", C.c_uint32),
                ("num_channels", C.c_uint16), ("num_samples", C.c_uint32),
                ("sampling_rate", C.c_uint32), ("bits_per_sample", C.c_uint16),
                ("num_samples_per_block", C.c_uint32), ("preset", C.c_uint8),
                ("ch_process_method", C.c_int)]


class LINNEEncodeParameter(C.Structure):
    _fields_ = [("num_channels", C.c_uint16), ("bits_per_sample", C.c_uint16),
                ("sampling_rate", C.c_uint32), ("num_samples_per_block", C.c_uint16),
                ("preset", C.c_uint8), ("ch_process_method", C.c_int),
                ("enable_learning", C.c_uint8), ("num_afmethod_iterations", C.c_uint8)]


class LINNEEncoderConfig(C.Structure):
    _fields_ = [("max_num_channels", C.c_uint32), ("max_num_samples_per_block", C.c_uint32),
                ("max_num_layers", C.c_uint32), ("max_num_parameters_per_layer", C.c_uint32)]


class LINNEDecoderConfig(C.Structure):
    _fields_ = [("max_num_channels", C.c_uint32), ("max_num_layers", C.c_uint32),
                ("max_num_parameters_per_layer", C.c_uint32), ("check_crc", C.c_uint8)]


def bind_linne_api(lib):
    """Declare argtypes/restype of the 14 public entry points on a loaded library."""
    u8p, u32p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32)
    i32pp = C.POINTER(C.POINTER(C.c_int32))
    lib.LINNEEncoder_EncodeHeader.argtypes = [C.POINTER(LINNEHeader), u8p, C.c_uint32]
    lib.LINNEEncoder_EncodeHeader.restype = C.c_int
    lib.LINNEEncoder_CalculateWorkSize.argtypes = [C.POINTER(LINNEEncoderConfig)]
    lib.LINNEEncoder_CalculateWorkSize.restype = C.c_int32
    lib.LINNEEncoder_Create.argtypes = [C.POINTER(LINNEEncoderConfig), C.c_void_p, C.c_int32]
    lib.LINNEEncoder_Create.restype = C.c_void_p
    lib.LINNEEncoder_Destroy.argtypes = [C.c_void_p]
    lib.LINNEEncoder_Destroy.restype = None
    lib.LINNEEncoder_SetEncodeParameter.argtypes = [C.c_void_p, C.POINTER(LINNEEncodeParameter)]
    lib.LINNEEncoder_SetEncodeParameter.restype = C.c_int
    for name in ("LINNEEncoder_EncodeBlock", "LINNEEncoder_EncodeWhole"):
        f = getattr(lib, name)
        f.argtypes = [C.c_void_p, i32pp, C.c_uint32, u8p, C.c_uint32, u32p]
        f.restype = C.c_int
    lib.LINNEDecoder_DecodeHeader.argtypes = [u8p, C.c_uint32, C.POINTER(LINNEHeader)]
    lib.LINNEDecoder_DecodeHeader.restype = C.c_int
    lib.LINNEDecoder_CalculateWorkSize.argtypes = [C.POINTER(LINNEDecoderConfig)]
    lib.LINNEDecoder_CalculateWorkSize.restype = C.c_int32
    lib.LINNEDecoder_Create.argtypes = [C.POINTER(LINNEDecoderConfig), C.c_void_p, C.c_int32]
    lib.LINNEDecoder_Create.restype = C.c_void_p
    lib.LINNEDecoder_Destroy.argtypes = [C.c_void_p]
    lib.LINNEDecoder_Destroy.restype = None
    lib.LINNEDecoder_SetHeader.argtypes = [C.c_void_p, C.POINTER(LINNEHeader)]
    lib.LINNEDecoder_SetHeader.restype = C.c_int
    lib.LINNEDecoder_DecodeBlock.argtypes = [C.c_void_p, u8p, C.c_uint32, i32pp, C.c_uint32,
                                             C.c_uint32, u32p, u32p]
    lib.LINNEDecoder_DecodeBlock.restype = C.c_int
    lib.LINNEDecoder_DecodeWhole.argtypes = [C.c_void_p, u8p, C.c_uint32, i32pp, C.c_uint32, C.c_uint32]
    lib.LINNEDecoder_DecodeWhole.restype = C.c_int
    return lib


def _chan_ptrs(pcm: np.ndarray):
    """pcm: int32 [C][n] C-contiguous -> (int32**) array of row pointers (keeps pcm alive by ref)."""
    assert pcm.dtype == np.int32 and pcm.ndim == 2 and pcm.flags["C_CONTIGUOUS"]
    arr = (C.POINTER(C.c_int32) * pcm.shape[0])()
    for c in range(pcm.shape[0]):
        arr[c] = pcm[c].ctypes.data_as(C.POINTER(C.c_int32))
    return arr


class LinneApi:
    """Drives any library exporting the LINNE public C API (reference or product)."""

    def __init__(self, lib):
        self.lib = bind_linne_api(lib)

    # -- encode ---------------------------------------------------------------------------------
    def make_encoder(self, channels, block, layers=3, params=128):
        cfg = LINNEEncoderConfig(channels, block, layers, params)
        h = self.lib.LINNEEncoder_Create(C.byref(cfg), None, 0)
        if not h:
            raise RuntimeError("LINNEEncoder_Create failed")
        return h

    def encode(self, pcm, bits=16, rate=44100, block=10240, preset=0, ms=None, learning=0, af=0,
               max_block=None, cap=None, whole=True, return_code=False):
        pcm = np.ascontiguousarray(pcm, dtype=np.int32)
        nch, n = pcm.shape
        if ms is None:
            ms = 1 if nch >= 2 else 0
        enc = self.make_encoder(nch, max_block or block)
        try:
            prm = LINNEEncodeParameter(nch, bits, rate, block, preset, ms, learning, af)
            rc = self.lib.LINNEEncoder_SetEncodeParameter(enc, C.byref(prm))
            if rc != OK:
                if return_code:
                    return rc, b""
                raise RuntimeError(f"SetEncodeParameter rc={rc}")
            if cap is None:
                cap = 30 + 2 * nch * n * 4 + 1024 * (n // block + 2)
            out = np.zeros(cap + 64, dtype=np.uint8)
            size = C.c_uint32(0)
            ptrs = _chan_ptrs(pcm)
            if whole:
                rc = self.lib.LINNEEncoder_EncodeWhole(enc, ptrs, n, out.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                       cap, C.byref(size))
            else:  # the CLI's loop: header + EncodeBlock per block (tools/linne_codec/linne_codec.c:123-161)
                hdr = LINNEHeader(1, 2, nch, n, rate, bits, block, preset, ms)
                rc = self.lib.LINNEEncoder_EncodeHeader(C.byref(hdr), out.ctypes.data_as(C.POINTER(C.c_uint8)), cap)
                off, done = 30, 0
                while rc == OK and done < n:
                    m = min(block, n - done)
                    sub = (C.POINTER(C.c_int32) * nch)()
                    for c in range(nch):
                        sub[c] = C.cast(pcm[c].ctypes.data + 4 * done, C.POINTER(C.c_int32))
                    rc = self.lib.LINNEEncoder_EncodeBlock(
                        enc, sub, m, C.cast(out.ctypes.data + off, C.POINTER(C.c_uint8)), cap - off, C.byref(size))
                    off += size.value
                    done += m
                size = C.c_uint32(off)
            if return_code:
                return rc, out[:size.value].tobytes() if rc == OK else b""
            if rc != OK:
                raise RuntimeError(f"encode rc={rc}")
            return out[:size.value].tobytes()
        finally:
            self.lib.LINNEEncoder_Destroy(enc)

    # -- decode ---------------------------------------------------------------------------------
    def decode_header(self, data: bytes):
        buf = np.frombuffer(data, dtype=np.uint8)
        hdr = LINNEHeader()
        rc = self.lib.LINNEDecoder_DecodeHeader(buf.ctypes.data_as(C.POINTER(C.c_uint8)), len(data), C.byref(hdr))
        return rc, hdr

    def decode(self, data: bytes, check_crc=1, return_code=False, out_channels=None, out_samples=None,
               fill=0):
        rc, hdr = self.decode_header(data)
        if rc != OK:
            if return_code:
                return rc, None
            raise RuntimeError(f"DecodeHeader rc={rc}")
        nch = out_channels if out_channels is not None else hdr.num_channels
        n = out_samples if out_samples is not None else hdr.num_samples
        cfg = LINNEDecoderConfig(max(nch, hdr.num_channels, 1), 3, 128, check_crc)
        dec = self.lib.LINNEDecoder_Create(C.byref(cfg), None, 0)
        if not dec:
            raise RuntimeError("LINNEDecoder_Create failed")
        try:
            # pad the stream: the reference's reader may touch up to 3 bytes past the end (SURVEY A11)
            buf = np.zeros(len(data) + 16, dtype=np.uint8)
            buf[:len(data)] = np.frombuffer(data, dtype=np.uint8)
            out = np.full((max(nch, 1), max(n, 1)), fill, dtype=np.int32)
            rc = self.lib.LINNEDecoder_DecodeWhole(dec, buf.ctypes.data_as(C.POINTER(C.c_uint8)), len(data),
                                                   _chan_ptrs(out), nch, n)
            if return_code:
                return rc, out
            if rc != OK:
                raise RuntimeError(f"decode rc={rc}")
            return out
        finally:
            self.lib.LINNEDecoder_Destroy(dec)


    # -- random access (include/linne_b200.h: seek index, sample windows) ---------------------------
    def _open_decoder(self, channels, check_crc):
        cfg = LINNEDecoderConfig(max(channels, 1), 3, 128, check_crc)
        dec = self.lib.LINNEDecoder_Create(C.byref(cfg), None, 0)
        if not dec:
            raise RuntimeError("LINNEDecoder_Create failed")
        return dec

    def _build_index(self, dec, data: bytes):
        buf = np.frombuffer(data, dtype=np.uint8)
        u8p = buf.ctypes.data_as(C.POINTER(C.c_uint8))
        n = C.c_uint32(0)
        rc = self.lib.LINNEB200_DecoderBuildIndex(dec, u8p, None, len(data), None, 0, C.byref(n))
        if rc not in (OK, INSUFFICIENT_BUFFER) and n.value == 0:
            return rc, np.zeros((0, 2), np.uint32)
        pts = (SeekPoint * max(1, n.value))()
        rc = self.lib.LINNEB200_DecoderBuildIndex(dec, u8p, None, len(data), pts, n.value, C.byref(n))
        arr = np.frombuffer(bytes(pts), dtype=np.uint32).reshape(-1, 2)[:n.value].copy()
        return rc, arr

    def build_index(self, data: bytes, return_code=False):
        """-> uint32 [N, 2]: (first sample, byte offset) of every block (LINNEB200_DecoderBuildIndex)"""
        rc, hdr = self.decode_header(data)
        dec = self._open_decoder(hdr.num_channels if rc == OK else 1, 1)
        try:
            rc, arr = self._build_index(dec, data)
        finally:
            self.lib.LINNEDecoder_Destroy(dec)
        if return_code:
            return rc, arr
        if rc != OK:
            raise RuntimeError(f"BuildIndex rc={rc}")
        return arr

    def _windows(self, data: bytes, starts, lengths, index, check_crc, return_code, what, call):
        """Shared by decode_windows and decode_windows_packed: the handle, the index (built when none is given) and the
        windows laid out back to back.  `call(dec, hdr, pts, npts, wins, num_windows, offs)` -> (rc, results)."""
        starts, lengths = [int(s) for s in starts], [int(n) for n in lengths]
        if len(starts) != len(lengths):
            raise ValueError("starts and lengths differ in length")
        rc, hdr = self.decode_header(data)
        if rc != OK:
            if return_code:
                return rc, [], []
            raise RuntimeError(f"DecodeHeader rc={rc}")
        dec = self._open_decoder(hdr.num_channels, check_crc)
        try:
            if index is None:
                rc, index = self._build_index(dec, data)
                if rc != OK:
                    if return_code:
                        return rc, [], []
                    raise RuntimeError(f"BuildIndex rc={rc}")
            else:
                rc = self.lib.LINNEDecoder_SetHeader(dec, C.byref(hdr))
                if rc != OK:
                    raise RuntimeError(f"SetHeader rc={rc}")
            pts, npts = index_points(index)
            offs = np.concatenate([[0], np.cumsum(lengths, dtype=np.int64)]).astype(np.int64)
            wins = (Window * max(1, len(starts)))(*[Window(s, n, int(o), 0) for s, n, o in zip(starts, lengths, offs)])
            rc, res = call(dec, hdr, pts, npts, wins, len(starts), offs)
            status = [int(wins[w].status) for w in range(len(starts))]
            if return_code:
                return rc, res, status
            if rc != OK:
                raise RuntimeError(f"{what} rc={rc} (statuses {status})")
            return res
        finally:
            self.lib.LINNEDecoder_Destroy(dec)

    def decode_windows(self, data: bytes, starts, lengths, index=None, check_crc=1, return_code=False):
        """Samples [starts[w], starts[w] + lengths[w]) of every channel -> list of int32 [C][len] arrays
        (LINNEB200_DecodeWindows); with return_code: (rc, arrays, per-window statuses)."""
        def call(dec, hdr, pts, npts, wins, nw, offs):
            nch = hdr.num_channels
            out = np.zeros((max(nch, 1), max(int(offs[-1]), 1)), dtype=np.int32)
            buf = np.frombuffer(data, dtype=np.uint8)
            rc = self.lib.LINNEB200_DecodeWindows(dec, buf.ctypes.data_as(C.POINTER(C.c_uint8)), len(data), pts, npts,
                                                  wins, nw, _chan_ptrs(out), nch, out.shape[1])
            return rc, [out[:, offs[w]:offs[w + 1]] for w in range(nw)]
        return self._windows(data, starts, lengths, index, check_crc, return_code, "DecodeWindows", call)

    def decode_windows_packed(self, data: bytes, starts, lengths, index=None, check_crc=1, return_code=False):
        """Frames [starts[w], starts[w] + lengths[w]) -> list of bytes, each the window's WAV data-chunk bytes
        (interleaved little-endian samples, LINNEB200_DecodeWindowsPacked); with return_code: (rc, list, statuses)."""
        def call(dec, hdr, pts, npts, wins, nw, offs):
            frame = hdr.num_channels * (hdr.bits_per_sample // 8)
            total = int(offs[-1])
            out = np.zeros(max(total * frame, 1), dtype=np.uint8)
            buf = np.frombuffer(data, dtype=np.uint8)
            u8p = C.POINTER(C.c_uint8)
            rc = self.lib.LINNEB200_DecodeWindowsPacked(dec, buf.ctypes.data_as(u8p), len(data), pts, npts, wins, nw,
                                                        out.ctypes.data_as(u8p), total)
            return rc, [out[offs[w] * frame:offs[w + 1] * frame].tobytes() for w in range(nw)]
        return self._windows(data, starts, lengths, index, check_crc, return_code, "DecodeWindowsPacked", call)

    # -- salvage (include/linne_b200.h: LINNEB200_DecodeSalvage / DecodeSalvagePacked) ------------------------------------
    def _salvage(self, data: bytes, header, call):
        """The handle with the stream's header latched -- `header` (a LINNEHeader) when given, e.g. for a stream whose own
        header is damaged, else the image's -- then `call(dec, hdr, buf, damage, capacity, count)` -> (rc, output), run
        again with room for every record when the first run found more than it had room for."""
        if header is None:
            rc, header = self.decode_header(data)
            if rc != OK:
                return rc, None, []
        dec = self._open_decoder(header.num_channels, 1)
        try:
            rc = self.lib.LINNEDecoder_SetHeader(dec, C.byref(header))
            if rc != OK:
                return rc, None, []
            buf = np.frombuffer(data, dtype=np.uint8)
            cap, count = 64, C.c_uint32(0)
            while True:
                damage = (Damage * cap)()
                rc, out = call(dec, header, buf.ctypes.data_as(C.POINTER(C.c_uint8)), damage, cap, count)
                if count.value <= cap:
                    break
                cap = count.value
            records = [(d.first_sample, d.num_samples, d.byte_offset, d.byte_size, d.status) for d in damage[:count.value]]
            return rc, out, records
        finally:
            self.lib.LINNEDecoder_Destroy(dec)

    def decode_salvage(self, data: bytes, header=None):
        """Every intact block of a possibly damaged stream (LINNEB200_DecodeSalvage) -> (rc, int32 [C][N] planes, records),
        records = [(first_sample, num_samples, byte_offset, byte_size, status)]; samples inside a record are zero."""
        def call(dec, hdr, u8p, damage, cap, count):
            out = np.zeros((max(hdr.num_channels, 1), max(hdr.num_samples, 1)), dtype=np.int32)
            rc = self.lib.LINNEB200_DecodeSalvage(dec, u8p, len(data), _chan_ptrs(out), hdr.num_channels, hdr.num_samples,
                                                  damage, cap, C.byref(count))
            return rc, out[:, :hdr.num_samples]
        return self._salvage(data, header, call)

    def decode_salvage_packed(self, data: bytes, header=None):
        """The same as WAV data-chunk bytes (LINNEB200_DecodeSalvagePacked) -> (rc, bytes, records)."""
        def call(dec, hdr, u8p, damage, cap, count):
            nbytes = hdr.num_samples * hdr.num_channels * (hdr.bits_per_sample // 8)
            out = np.zeros(max(nbytes, 1), dtype=np.uint8)
            rc = self.lib.LINNEB200_DecodeSalvagePacked(dec, u8p, len(data), out.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                        hdr.num_samples, damage, cap, C.byref(count))
            return rc, out[:nbytes].tobytes()
        return self._salvage(data, header, call)


def bind_ext_api(lib):
    """Declare the LINNEB200_* extension entry points (include/linne_b200.h)."""
    lib.LINNEB200_Backend.restype = C.c_char_p
    lib.LINNEB200_DeviceAvailable.restype = C.c_int
    lib.LINNEB200_EncoderLaunchCount.argtypes = [C.c_void_p]
    lib.LINNEB200_EncoderLaunchCount.restype = C.c_uint64
    lib.LINNEB200_DecoderLaunchCount.argtypes = [C.c_void_p]
    lib.LINNEB200_DecoderLaunchCount.restype = C.c_uint64
    lib.LINNEB200_EncoderUseStream.argtypes = [C.c_void_p, C.c_void_p]
    lib.LINNEB200_DecoderUseStream.argtypes = [C.c_void_p, C.c_void_p]
    u8p, u32p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32)
    lib.LINNEB200_EncodeWholeResident.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32,
                                                  C.c_void_p, C.c_uint32, u32p]
    lib.LINNEB200_EncodeWholeResident.restype = C.c_int
    lib.LINNEB200_DecodeWholeResident.argtypes = [C.c_void_p, u8p, C.c_void_p, C.c_uint32, C.c_void_p,
                                                  C.c_uint32, C.c_uint32, C.c_uint32]
    lib.LINNEB200_DecodeWholeResident.restype = C.c_int
    lib.LINNEB200_EncodeWholeWithParams.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_int32)), C.c_uint32,
                                                    C.POINTER(ChannelParams), C.c_uint32, u8p, C.c_uint32, u32p]
    lib.LINNEB200_EncodeWholeWithParams.restype = C.c_int
    for side in ("Encoder", "Decoder"):
        getattr(lib, f"LINNEB200_{side}SetProfiling").argtypes = [C.c_void_p, C.c_int]
        getattr(lib, f"LINNEB200_{side}ResetStageStats").argtypes = [C.c_void_p]
        f = getattr(lib, f"LINNEB200_{side}GetStageStats")
        f.argtypes = [C.c_void_p, C.POINTER(StageStat), C.c_int]
        f.restype = C.c_int
    lib.LINNEB200_MeasureFp64Tflops.restype = C.c_double
    lib.LINNEB200_DeviceAlloc.argtypes = [C.c_size_t]
    lib.LINNEB200_DeviceAlloc.restype = C.c_void_p
    lib.LINNEB200_DeviceFree.argtypes = [C.c_void_p]
    lib.LINNEB200_IpcExport.argtypes = [C.c_void_p, u8p]
    lib.LINNEB200_IpcExport.restype = C.c_int
    lib.LINNEB200_IpcOpen.argtypes = [u8p]
    lib.LINNEB200_IpcOpen.restype = C.c_void_p
    lib.LINNEB200_IpcClose.argtypes = [C.c_void_p]
    lib.LINNEB200_EncodeWholePacked.argtypes = [C.c_void_p, u8p, C.c_uint32, u8p, C.c_uint32, u32p]
    lib.LINNEB200_EncodeWholePacked.restype = C.c_int
    lib.LINNEB200_DecodeWholePacked.argtypes = [C.c_void_p, u8p, C.c_uint32, u8p, C.c_uint32, u32p]
    lib.LINNEB200_DecodeWholePacked.restype = C.c_int
    lib.LINNEB200_EncodeFilesResident.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(FileDesc), C.c_uint32,
                                                  C.c_void_p, C.c_uint32, u32p]
    lib.LINNEB200_EncodeFilesResident.restype = C.c_int
    lib.LINNEB200_DecodeFilesResident.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(FileDesc), C.c_uint32,
                                                  C.c_void_p, C.c_uint32]
    lib.LINNEB200_DecodeFilesResident.restype = C.c_int
    lib.LINNEB200_EncodeFilesPacked.argtypes = [C.c_void_p, u8p, C.POINTER(FileDesc), C.c_uint32, u8p, C.c_uint32, u32p]
    lib.LINNEB200_EncodeFilesPacked.restype = C.c_int
    lib.LINNEB200_DecodeFilesPacked.argtypes = [C.c_void_p, u8p, C.c_uint32, C.POINTER(FileDesc), C.c_uint32, u8p]
    lib.LINNEB200_DecodeFilesPacked.restype = C.c_int
    lib.LINNEB200_DecoderBuildIndex.argtypes = [C.c_void_p, u8p, C.c_void_p, C.c_uint32, C.POINTER(SeekPoint), C.c_uint32, u32p]
    lib.LINNEB200_DecoderBuildIndex.restype = C.c_int
    lib.LINNEB200_DecodeWindows.argtypes = [C.c_void_p, u8p, C.c_uint32, C.POINTER(SeekPoint), C.c_uint32, C.POINTER(Window),
                                            C.c_uint32, C.POINTER(C.POINTER(C.c_int32)), C.c_uint32, C.c_uint32]
    lib.LINNEB200_DecodeWindows.restype = C.c_int
    lib.LINNEB200_DecodeWindowsResident.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(SeekPoint), C.c_uint32,
                                                    C.POINTER(Window), C.c_uint32, C.c_void_p, C.c_uint32]
    lib.LINNEB200_DecodeWindowsResident.restype = C.c_int
    lib.LINNEB200_DecodeWindowsPacked.argtypes = [C.c_void_p, u8p, C.c_uint32, C.POINTER(SeekPoint), C.c_uint32, C.POINTER(Window),
                                                  C.c_uint32, u8p, C.c_uint32]
    lib.LINNEB200_DecodeWindowsPacked.restype = C.c_int
    dmg = C.POINTER(Damage)
    lib.LINNEB200_DecodeSalvage.argtypes = [C.c_void_p, u8p, C.c_uint32, C.POINTER(C.POINTER(C.c_int32)), C.c_uint32, C.c_uint32,
                                            dmg, C.c_uint32, u32p]
    lib.LINNEB200_DecodeSalvage.restype = C.c_int
    lib.LINNEB200_DecodeSalvagePacked.argtypes = [C.c_void_p, u8p, C.c_uint32, u8p, C.c_uint32, dmg, C.c_uint32, u32p]
    lib.LINNEB200_DecodeSalvagePacked.restype = C.c_int
    lib.LINNEB200_DecoderSetReadahead.argtypes = [C.c_void_p, C.c_uint32]
    lib.LINNEB200_DecoderSetThroughputBlocks.argtypes = [C.c_void_p, C.c_uint32]
    lib.LINNEB200_EncoderSetDevices.argtypes = [C.c_void_p, C.c_uint32]
    lib.LINNEB200_DecoderSetDevices.argtypes = [C.c_void_p, C.c_uint32]
    lib.LINNEB200_HostAlloc.argtypes = [C.c_size_t]
    lib.LINNEB200_HostAlloc.restype = C.c_void_p
    lib.LINNEB200_HostFree.argtypes = [C.c_void_p]
    for name in ("DeviceCopy", "CopyToDevice", "CopyToHost"):
        f = getattr(lib, f"LINNEB200_{name}")
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        f.restype = C.c_int
    return lib


_lib = None


def load_library():
    """Load liblinne_b200.so (built in-tree by __graft_entry__.build() / make -C linne_b200/csrc product)."""
    global _lib
    if _lib is None:
        if not os.path.exists(PRODUCT_SO):
            raise RuntimeError(
                f"{PRODUCT_SO} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "linne_b200 has no CPU fallback.")
        lib = C.CDLL(PRODUCT_SO, mode=getattr(os, "RTLD_LOCAL", 0))
        bind_linne_api(lib)
        bind_ext_api(lib)
        _lib = lib
    return _lib


class StageStat(C.Structure):
    _fields_ = [("name", C.c_char * 24), ("launches", C.c_uint64), ("total_ms", C.c_double)]


class TimelineEntry(C.Structure):
    _fields_ = [("name", C.c_char * 24), ("begin_ms", C.c_float), ("end_ms", C.c_float)]


class FileDesc(C.Structure):
    """struct LINNEB200FileDesc (include/linne_b200.h)"""
    _fields_ = [("first_sample", C.c_uint32), ("num_samples", C.c_uint32), ("out_offset", C.c_uint32),
                ("out_size", C.c_uint32), ("status", C.c_int32)]


class SeekPoint(C.Structure):
    """struct LINNEB200SeekPoint (include/linne_b200.h): one block of a seek index"""
    _fields_ = [("first_sample", C.c_uint32), ("byte_offset", C.c_uint32)]


class Window(C.Structure):
    """struct LINNEB200Window (include/linne_b200.h): one sample window of LINNEB200_DecodeWindows"""
    _fields_ = [("first_sample", C.c_uint32), ("num_samples", C.c_uint32), ("out_offset", C.c_uint32), ("status", C.c_int32)]


class Damage(C.Structure):
    """struct LINNEB200Damage (include/linne_b200.h): one run of samples a salvage decode could not recover"""
    _fields_ = [("first_sample", C.c_uint32), ("num_samples", C.c_uint32), ("byte_offset", C.c_uint32),
                ("byte_size", C.c_uint32), ("status", C.c_int32)]


def index_points(index):
    """uint32 [N, 2] (first_sample, byte_offset) -> ctypes SeekPoint array"""
    index = np.ascontiguousarray(index, dtype=np.uint32).reshape(-1, 2)
    return (SeekPoint * max(1, len(index))).from_buffer_copy(index.tobytes() or bytes(8)), len(index)


class ChannelParams(C.Structure):
    """struct LINNEB200ChannelParams (include/linne_b200.h)"""
    _fields_ = [("log2_units", C.c_uint8 * 3), ("rshift", C.c_uint8 * 3), ("coef", (C.c_int8 * 128) * 3)]


class _Session:
    """A long-lived encoder or decoder handle (what a server keeps per stream/worker)."""
    _side = ""

    def __init__(self, lib, handle):
        self.lib, self.h = lib, handle

    def use_stream(self, cuda_stream_ptr):
        getattr(self.lib, f"LINNEB200_{self._side}UseStream")(self.h, C.c_void_p(cuda_stream_ptr))

    def set_profiling(self, on=True):
        getattr(self.lib, f"LINNEB200_{self._side}SetProfiling")(self.h, 1 if on else 0)

    def reset_stage_stats(self):
        getattr(self.lib, f"LINNEB200_{self._side}ResetStageStats")(self.h)

    def stage_stats(self):
        buf = (StageStat * 32)()
        n = getattr(self.lib, f"LINNEB200_{self._side}GetStageStats")(self.h, buf, 32)
        return {buf[i].name.decode(): (int(buf[i].launches), float(buf[i].total_ms)) for i in range(n)}

    def timeline(self):
        """[(kernel, begin_ms, end_ms)] since the process-wide origin, for the launches profiled since the last reset."""
        buf = (TimelineEntry * 2048)()
        f = getattr(self.lib, f"LINNEB200_{self._side}GetTimeline")
        f.argtypes = [C.c_void_p, C.POINTER(TimelineEntry), C.c_int]
        f.restype = C.c_int
        n = f(self.h, buf, 2048)
        return [(buf[i].name.decode(), float(buf[i].begin_ms), float(buf[i].end_ms)) for i in range(n)]

    def launch_count(self):
        return int(getattr(self.lib, f"LINNEB200_{self._side}LaunchCount")(self.h))

    def set_devices(self, n):
        """shard the whole-stream calls of this handle over n block ranges / devices (include/linne_b200.h)"""
        getattr(self.lib, f"LINNEB200_{self._side}SetDevices")(self.h, int(n))

    def close(self):
        if self.h:
            getattr(self.lib, f"LINNE{self._side}_Destroy")(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EncoderSession(_Session):
    _side = "Encoder"

    def __init__(self, channels, bits=16, rate=44100, block=10240, preset=0, ms=None, learning=0, af=0,
                 max_block=None, lib=None):
        lib = lib or load_library()
        cfg = LINNEEncoderConfig(channels, max_block or block, 3, 128)
        h = lib.LINNEEncoder_Create(C.byref(cfg), None, 0)
        if not h:
            raise RuntimeError("LINNEEncoder_Create failed (no CUDA device? linne_b200 has no CPU fallback)")
        super().__init__(lib, h)
        if ms is None:
            ms = 1 if channels >= 2 else 0
        prm = LINNEEncodeParameter(channels, bits, rate, block, preset, ms, learning, af)
        rc = lib.LINNEEncoder_SetEncodeParameter(h, C.byref(prm))
        if rc != OK:
            raise RuntimeError(f"SetEncodeParameter rc={rc}")
        self.channels = channels

    def encode_whole(self, chan_ptrs, n, out_ptr, cap):
        """chan_ptrs: (int32*)[C] ctypes array of host pointers; out_ptr: host address. Returns bytes written."""
        size = C.c_uint32(0)
        rc = self.lib.LINNEEncoder_EncodeWhole(self.h, chan_ptrs, n, C.cast(out_ptr, C.POINTER(C.c_uint8)), cap, C.byref(size))
        if rc != OK:
            raise RuntimeError(f"EncodeWhole rc={rc}")
        return size.value

    def encode_whole_resident(self, d_pcm_ptr, stride, n, d_out_ptr, cap):
        size = C.c_uint32(0)
        rc = self.lib.LINNEB200_EncodeWholeResident(self.h, C.c_void_p(d_pcm_ptr), stride, n, C.c_void_p(d_out_ptr), cap, C.byref(size))
        if rc != OK:
            raise RuntimeError(f"EncodeWholeResident rc={rc}")
        return size.value


class DecoderSession(_Session):
    _side = "Decoder"

    def __init__(self, channels=8, check_crc=1, lib=None):
        lib = lib or load_library()
        cfg = LINNEDecoderConfig(channels, 3, 128, check_crc)
        h = lib.LINNEDecoder_Create(C.byref(cfg), None, 0)
        if not h:
            raise RuntimeError("LINNEDecoder_Create failed (no CUDA device? linne_b200 has no CPU fallback)")
        super().__init__(lib, h)

    def decode_whole(self, data_ptr, size, chan_ptrs, channels, n):
        rc = self.lib.LINNEDecoder_DecodeWhole(self.h, C.cast(data_ptr, C.POINTER(C.c_uint8)), size, chan_ptrs, channels, n)
        if rc != OK:
            raise RuntimeError(f"DecodeWhole rc={rc}")

    def decode_whole_resident(self, data_ptr, d_data_ptr, size, d_pcm_ptr, stride, channels, n):
        host = C.cast(data_ptr, C.POINTER(C.c_uint8)) if data_ptr else None
        rc = self.lib.LINNEB200_DecodeWholeResident(self.h, host, C.c_void_p(d_data_ptr),
                                                    size, C.c_void_p(d_pcm_ptr), stride, channels, n)
        if rc != OK:
            raise RuntimeError(f"DecodeWholeResident rc={rc}")


class DeviceBuffer:
    """Raw device memory of the current CUDA device (LINNEB200_DeviceAlloc): exportable to peer processes."""

    def __init__(self, nbytes, lib=None):
        self.lib = lib or load_library()
        self.nbytes = int(nbytes)
        self.ptr = self.lib.LINNEB200_DeviceAlloc(self.nbytes)
        if not self.ptr:
            raise MemoryError(f"LINNEB200_DeviceAlloc({nbytes}) failed")

    def ipc_handle(self) -> bytes:
        h = (C.c_uint8 * 64)()
        if self.lib.LINNEB200_IpcExport(C.c_void_p(self.ptr), h) != 0:
            raise RuntimeError("LINNEB200_IpcExport failed")
        return bytes(h)

    def upload(self, data: bytes, offset=0):
        buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
        if self.lib.LINNEB200_CopyToDevice(C.c_void_p(self.ptr + offset), buf, len(data)) != 0:
            raise RuntimeError("LINNEB200_CopyToDevice failed")

    def download(self, nbytes=None, offset=0) -> bytes:
        n = self.nbytes - offset if nbytes is None else int(nbytes)
        buf = (C.c_uint8 * n)()
        if self.lib.LINNEB200_CopyToHost(buf, C.c_void_p(self.ptr + offset), n) != 0:
            raise RuntimeError("LINNEB200_CopyToHost failed")
        return bytes(buf)

    def free(self):
        if self.ptr:
            self.lib.LINNEB200_DeviceFree(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PeerMapping:
    """A peer process's DeviceBuffer mapped into this process (CUDA IPC; copies run over NVLink)."""

    def __init__(self, handle: bytes, lib=None):
        self.lib = lib or load_library()
        h = (C.c_uint8 * 64).from_buffer_copy(handle)
        self.ptr = self.lib.LINNEB200_IpcOpen(h)
        if not self.ptr:
            raise RuntimeError("LINNEB200_IpcOpen failed (no peer access between these devices?)")

    def put(self, offset, d_src_ptr, nbytes):
        """device -> peer device copy of `nbytes` from local device address `d_src_ptr`."""
        if self.lib.LINNEB200_DeviceCopy(C.c_void_p(self.ptr + offset), C.c_void_p(d_src_ptr), nbytes) != 0:
            raise RuntimeError("LINNEB200_DeviceCopy to the peer failed")

    def close(self):
        if self.ptr:
            self.lib.LINNEB200_IpcClose(C.c_void_p(self.ptr))
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Product(LinneApi):
    """The CUDA product behind the reference API."""

    def __init__(self):
        super().__init__(load_library())
        if self.lib.LINNEB200_Backend() != b"cuda-sm_100a":
            raise RuntimeError("liblinne_b200.so is not the CUDA build")

    def device_available(self) -> bool:
        return bool(self.lib.LINNEB200_DeviceAvailable())

    def measure_fp64_tflops(self) -> float:
        return float(self.lib.LINNEB200_MeasureFp64Tflops())

    def encode_packed(self, packed: bytes, channels, bits=16, rate=44100, block=10240, preset=0, ms=None, return_code=False):
        """`packed`: interleaved little-endian PCM as in a WAV data chunk (LINNEB200_EncodeWholePacked)."""
        u8p = C.POINTER(C.c_uint8)
        nbytes = bits // 8
        n = len(packed) // (channels * nbytes)
        if ms is None:
            ms = 1 if channels >= 2 else 0
        enc = self.make_encoder(channels, block)
        try:
            prm = LINNEEncodeParameter(channels, bits, rate, block, preset, ms, 0, 0)
            rc = self.lib.LINNEEncoder_SetEncodeParameter(enc, C.byref(prm))
            if rc != OK:
                raise RuntimeError(f"SetEncodeParameter rc={rc}")
            cap = 30 + 2 * channels * n * 4 + 4096
            out = np.zeros(cap, dtype=np.uint8)
            src = np.frombuffer(packed, dtype=np.uint8)
            size = C.c_uint32(0)
            rc = self.lib.LINNEB200_EncodeWholePacked(enc, src.ctypes.data_as(u8p), n, out.ctypes.data_as(u8p), cap, C.byref(size))
            if return_code:
                return rc, out[:size.value].tobytes() if rc == OK else b""
            if rc != OK:
                raise RuntimeError(f"EncodeWholePacked rc={rc}")
            return out[:size.value].tobytes()
        finally:
            self.lib.LINNEEncoder_Destroy(enc)

    def decode_packed(self, data: bytes, check_crc=1, return_code=False):
        """-> interleaved little-endian PCM bytes (LINNEB200_DecodeWholePacked)."""
        u8p = C.POINTER(C.c_uint8)
        rc, hdr = self.decode_header(data)
        if rc != OK:
            raise RuntimeError(f"DecodeHeader rc={rc}")
        cfg = LINNEDecoderConfig(8, 3, 128, check_crc)
        dec = self.lib.LINNEDecoder_Create(C.byref(cfg), None, 0)
        if not dec:
            raise RuntimeError("LINNEDecoder_Create failed")
        try:
            nbytes = hdr.bits_per_sample // 8
            out = np.zeros(max(1, hdr.num_samples * hdr.num_channels * nbytes), dtype=np.uint8)
            buf = np.frombuffer(data, dtype=np.uint8)
            frames = C.c_uint32(0)
            rc = self.lib.LINNEB200_DecodeWholePacked(dec, buf.ctypes.data_as(u8p), len(data), out.ctypes.data_as(u8p),
                                                      hdr.num_samples, C.byref(frames))
            res = out[:frames.value * hdr.num_channels * nbytes].tobytes()
            if return_code:
                return rc, res
            if rc != OK:
                raise RuntimeError(f"DecodeWholePacked rc={rc}")
            return res
        finally:
            self.lib.LINNEDecoder_Destroy(dec)

    def encode_with_params(self, pcm, params, bits=16, rate=44100, block=10240, preset=0, ms=None, return_code=False):
        """params: ctypes array of ChannelParams, one per (block, channel), block-major."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int32)
        nch, n = pcm.shape
        sess = EncoderSession(nch, bits=bits, rate=rate, block=block, preset=preset, ms=ms, lib=self.lib)
        try:
            cap = 30 + 2 * nch * n * 4 + 4096
            out = np.zeros(cap, dtype=np.uint8)
            size = C.c_uint32(0)
            rc = self.lib.LINNEB200_EncodeWholeWithParams(sess.h, _chan_ptrs(pcm), n, params, len(params) // nch,
                                                          out.ctypes.data_as(C.POINTER(C.c_uint8)), cap, C.byref(size))
            if return_code:
                return rc, out[:size.value].tobytes() if rc == OK else b""
            if rc != OK:
                raise RuntimeError(f"EncodeWholeWithParams rc={rc}")
            return out[:size.value].tobytes()
        finally:
            sess.close()
