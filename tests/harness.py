"""Shared test/bench harness: ctypes bindings and synthetic PCM generators.

Three libraries can be driven through the *same* LINNE C API shape:
  * the product      linne_b200/liblinne_b200.so         (CUDA, sm_100a)      -> linne_b200.api
  * the reference    oracle/_ref/liblinne_ref.so         (unmodified C, built by oracle/Makefile)
  * the oracle port  oracle/liblinne_oracle.so           (our plain-C restatement)

The reference and the oracle are CHECKERS: only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs import this module's `Ref` / `Oracle` classes.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from linne_b200.api import (LINNEHeader, LINNEEncodeParameter, LINNEEncoderConfig, LINNEDecoderConfig,  # noqa: E402
                            bind_linne_api, LinneApi, _chan_ptrs, PRESET_LAYERS)
REF_SO = os.path.join(ROOT, "oracle", "_ref", "liblinne_ref.so")
ORACLE_SO = os.path.join(ROOT, "oracle", "liblinne_oracle.so")

OK, INVALID_ARGUMENT, INVALID_FORMAT, INSUFFICIENT_BUFFER, INSUFFICIENT_DATA, \
    PARAMETER_NOT_SET, DATA_CORRUPTION, NG = range(8)


# ----------------------------------------------------------------------------------------------
# The unmodified reference (oracle/_ref) with the probe entry points of oracle/ref_probe.c
# ----------------------------------------------------------------------------------------------
def have_ref() -> bool:
    return os.path.exists(REF_SO)


class Ref(LinneApi):
    def __init__(self):
        super().__init__(C.CDLL(REF_SO, mode=getattr(os, "RTLD_LOCAL", 0)))
        L = self.lib
        L.RefProbe_EncoderLastParams.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32),
                                                 C.POINTER(C.c_uint32), C.POINTER(C.c_int32), C.c_uint32]
        L.RefProbe_EncoderLastPreemphasis.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        L.RefProbe_EncoderLastResidual.argtypes = [C.c_void_p, C.c_uint32]
        L.RefProbe_EncoderLastResidual.restype = C.POINTER(C.c_int32)
        L.RefProbe_CRC16.argtypes = [C.POINTER(C.c_uint8), C.c_uint64]
        L.RefProbe_CRC16.restype = C.c_uint16
        L.RefProbe_HuffmanCodes.argtypes = [C.POINTER(C.c_uint32), C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint8)]
        L.RefProbe_QuantizeCoefficients.argtypes = [C.POINTER(C.c_double), C.c_uint32, C.POINTER(C.c_int32), C.POINTER(C.c_uint32)]

    def crc16(self, data: bytes) -> int:
        buf = np.frombuffer(data, dtype=np.uint8)
        return int(self.lib.RefProbe_CRC16(buf.ctypes.data_as(C.POINTER(C.c_uint8)), len(data)))

    def huffman_codes(self, counts):
        cnt = np.asarray(counts, dtype=np.uint32)
        codes = np.zeros(len(cnt), dtype=np.uint32)
        lens = np.zeros(len(cnt), dtype=np.uint8)
        self.lib.RefProbe_HuffmanCodes(cnt.ctypes.data_as(C.POINTER(C.c_uint32)), len(cnt),
                                       codes.ctypes.data_as(C.POINTER(C.c_uint32)),
                                       lens.ctypes.data_as(C.POINTER(C.c_uint8)))
        return codes, lens

    def encode_blocks_traced(self, pcm, bits=16, rate=44100, block=10240, preset=0, ms=None, learning=0, af=0):
        """Encode block by block; returns (stream bytes, [per-block dict with type, bytes, per-channel
        params: units/rshift/coef/preem]) -- the reference's analysis results for the
        'identical coefficients -> identical bytes' leg."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int32)
        nch, n = pcm.shape
        if ms is None:
            ms = 1 if nch >= 2 else 0
        layers = PRESET_LAYERS[preset]
        enc = self.make_encoder(nch, block)
        try:
            prm = LINNEEncodeParameter(nch, bits, rate, block, preset, ms, learning, af)
            assert self.lib.LINNEEncoder_SetEncodeParameter(enc, C.byref(prm)) == OK
            cap = 11 + 2 * nch * block * 4 + 4096
            out = np.zeros(cap, dtype=np.uint8)
            hdr = LINNEHeader(1, 2, nch, n, rate, bits, block, preset, ms)
            hbuf = np.zeros(30, dtype=np.uint8)
            assert self.lib.LINNEEncoder_EncodeHeader(C.byref(hdr), hbuf.ctypes.data_as(C.POINTER(C.c_uint8)), 30) == OK
            stream = [hbuf.tobytes()]
            blocks = []
            done = 0
            while done < n:
                m = min(block, n - done)
                sub = (C.POINTER(C.c_int32) * nch)()
                for c in range(nch):
                    sub[c] = C.cast(pcm[c].ctypes.data + 4 * done, C.POINTER(C.c_int32))
                size = C.c_uint32(0)
                rc = self.lib.LINNEEncoder_EncodeBlock(enc, sub, m, out.ctypes.data_as(C.POINTER(C.c_uint8)), cap, C.byref(size))
                assert rc == OK, rc
                blk = out[:size.value].tobytes()
                info = {"type": blk[8], "nsamples": m, "bytes": blk, "channels": []}
                if blk[8] == 0:
                    for c in range(nch):
                        chd = {"units": [], "rshift": [], "coef": []}
                        for l, P in enumerate(layers):
                            u, r = C.c_uint32(0), C.c_uint32(0)
                            q = np.zeros(P, dtype=np.int32)
                            self.lib.RefProbe_EncoderLastParams(enc, c, l, C.byref(u), C.byref(r),
                                                                q.ctypes.data_as(C.POINTER(C.c_int32)), P)
                            chd["units"].append(u.value); chd["rshift"].append(r.value); chd["coef"].append(q)
                        prev = (C.c_int32 * 2)(); pc = (C.c_int32 * 2)()
                        self.lib.RefProbe_EncoderLastPreemphasis(enc, c, prev, pc)
                        chd["preem_prev"] = [prev[0], prev[1]]; chd["preem_coef"] = [pc[0], pc[1]]
                        rp = self.lib.RefProbe_EncoderLastResidual(enc, c)
                        chd["residual"] = np.ctypeslib.as_array(rp, shape=(m,)).copy()
                        info["channels"].append(chd)
                blocks.append(info)
                stream.append(blk)
                done += m
            return b"".join(stream), blocks
        finally:
            self.lib.LINNEEncoder_Destroy(enc)


# ----------------------------------------------------------------------------------------------
# The reference's answers for the inputs of the comparison tests, stored in tests/golden/reference_record.json
# (made by tests/golden/make_golden.py --record), so that a checkout without oracle/_ref still compares
# ----------------------------------------------------------------------------------------------
RECORD_JSON = os.path.join(ROOT, "tests", "golden", "reference_record.json")


def digest(data: bytes) -> str:
    """A stream as it is recorded: its length and SHA-256."""
    return f"{len(data)}:{hashlib.sha256(data).hexdigest()}"


class ReferenceRecord:
    """expect(key, ask) is what the reference answers to `ask`.  With a live reference (`live`, where oracle/_ref was
    built) the answer is ask(live) and must equal the stored one; without it the stored answer stands in.  With
    `recording` set, answers are taken from `live` and collected in `answers` instead of checked."""

    def __init__(self, live=None, recording=False):
        self.live, self.recording, self.answers = live, recording, {}
        if not recording:
            with open(RECORD_JSON) as f:
                self.stored = json.load(f)["answers"]

    def expect(self, key, ask):
        if self.recording:
            self.answers[key] = ask(self.live)
            return self.answers[key]
        assert key in self.stored, f"{key} is not in {os.path.relpath(RECORD_JSON, ROOT)}"
        want = self.stored[key]
        if self.live is not None:
            assert ask(self.live) == want, f"the reference's answer to {key} differs from the stored one"
        return want


# ----------------------------------------------------------------------------------------------
# Our plain-C restatement (oracle/liblinne_oracle.so)
# ----------------------------------------------------------------------------------------------
class LoChannelTrace(C.Structure):
    _fields_ = [("preem_prev", C.c_int32 * 2), ("preem_coef", C.c_int32 * 2),
                ("num_units", C.c_uint32 * 3), ("rshift", C.c_uint32 * 3),
                ("coef", (C.c_int32 * 128) * 3), ("coef_f64", (C.c_double * 128) * 3),
                ("porder", C.c_uint32), ("residual_bits", C.c_uint32)]


class Oracle:
    def __init__(self):
        L = self.lib = C.CDLL(ORACLE_SO, mode=getattr(os, "RTLD_LOCAL", 0))
        u8p, u32p = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32)
        i32pp = C.POINTER(C.POINTER(C.c_int32))
        L.lo_crc16.argtypes = [u8p, C.c_size_t]; L.lo_crc16.restype = C.c_uint16
        L.lo_huffman_build.argtypes = [u32p, C.c_uint32, u32p, u8p]
        L.lo_coef_huffman_table.argtypes = [u32p, u8p]
        L.lo_rice_parameter.argtypes = [C.c_double, u32p, u32p]
        L.lo_encoder_create.argtypes = [C.c_uint32, C.c_uint32]; L.lo_encoder_create.restype = C.c_void_p
        L.lo_encoder_destroy.argtypes = [C.c_void_p]
        L.lo_encoder_configure.argtypes = [C.c_void_p] + [C.c_uint32] * 8
        L.lo_encode_whole.argtypes = [C.c_void_p, i32pp, C.c_uint32, u8p, C.c_uint32, u32p]
        L.lo_encode_block.argtypes = [C.c_void_p, i32pp, C.c_uint32, u8p, C.c_uint32, u32p]
        L.lo_encode_block_forced.argtypes = [C.c_void_p, i32pp, C.c_uint32, C.POINTER(LoChannelTrace), u8p, C.c_uint32, u32p]
        L.lo_encoder_trace.argtypes = [C.c_void_p, C.c_uint32]; L.lo_encoder_trace.restype = C.POINTER(LoChannelTrace)
        L.lo_encoder_last_residual.argtypes = [C.c_void_p, C.c_uint32]
        L.lo_encoder_last_residual.restype = C.POINTER(C.c_int32)
        L.lo_encoder_last_block_type.argtypes = [C.c_void_p]
        L.lo_decode_whole.argtypes = [u8p, C.c_uint32, C.c_int, i32pp, C.c_uint32, C.c_uint32]
        L.lo_quantize.argtypes = [C.POINTER(C.c_double), C.c_uint32, C.POINTER(C.c_int32), u32p]
        L.lo_coder_plan.argtypes = [C.POINTER(C.c_int32), C.c_uint32, u32p, u32p]
        L.lo_coder_plan.restype = C.c_uint32

    def crc16(self, data: bytes) -> int:
        buf = np.frombuffer(data, dtype=np.uint8)
        return int(self.lib.lo_crc16(buf.ctypes.data_as(C.POINTER(C.c_uint8)), len(data)))

    def huffman_codes(self, counts):
        cnt = np.asarray(counts, dtype=np.uint32)
        codes = np.zeros(len(cnt), dtype=np.uint32)
        lens = np.zeros(len(cnt), dtype=np.uint8)
        self.lib.lo_huffman_build(cnt.ctypes.data_as(C.POINTER(C.c_uint32)), len(cnt),
                                  codes.ctypes.data_as(C.POINTER(C.c_uint32)), lens.ctypes.data_as(C.POINTER(C.c_uint8)))
        return codes, lens

    def coef_table(self):
        codes = np.zeros(256, dtype=np.uint32); lens = np.zeros(256, dtype=np.uint8)
        self.lib.lo_coef_huffman_table(codes.ctypes.data_as(C.POINTER(C.c_uint32)), lens.ctypes.data_as(C.POINTER(C.c_uint8)))
        return codes, lens

    def rice_k2(self, mean: float) -> int:
        k1, k2 = C.c_uint32(0), C.c_uint32(0)
        self.lib.lo_rice_parameter(mean, C.byref(k1), C.byref(k2))
        return k2.value

    def encode(self, pcm, bits=16, rate=44100, block=10240, preset=0, ms=None, learning=0, af=0,
               max_block=None, cap=None, return_code=False):
        pcm = np.ascontiguousarray(pcm, dtype=np.int32)
        nch, n = pcm.shape
        if ms is None:
            ms = 1 if nch >= 2 else 0
        enc = self.lib.lo_encoder_create(nch, max_block or block)
        try:
            rc = self.lib.lo_encoder_configure(enc, nch, bits, rate, block, preset, ms, learning, af)
            if rc != OK:
                if return_code:
                    return rc, b""
                raise RuntimeError(f"configure rc={rc}")
            if cap is None:
                cap = 30 + 2 * nch * n * 4 + 1024 * (n // block + 2)
            out = np.zeros(cap, dtype=np.uint8)
            size = C.c_uint32(0)
            rc = self.lib.lo_encode_whole(enc, _chan_ptrs(pcm), n, out.ctypes.data_as(C.POINTER(C.c_uint8)), cap, C.byref(size))
            if return_code:
                return rc, out[:size.value].tobytes() if rc == OK else b""
            if rc != OK:
                raise RuntimeError(f"encode rc={rc}")
            return out[:size.value].tobytes()
        finally:
            self.lib.lo_encoder_destroy(enc)

    def decode(self, data: bytes, check_crc=1, return_code=False):
        buf = np.frombuffer(data, dtype=np.uint8)
        nch = int.from_bytes(data[12:14], "big"); n = int.from_bytes(data[14:18], "big")
        out = np.zeros((max(nch, 1), max(n, 1)), dtype=np.int32)
        rc = self.lib.lo_decode_whole(buf.ctypes.data_as(C.POINTER(C.c_uint8)), len(data), check_crc,
                                      _chan_ptrs(out), nch, n)
        if return_code:
            return rc, out
        if rc != OK:
            raise RuntimeError(f"decode rc={rc}")
        return out


# ----------------------------------------------------------------------------------------------
# Synthetic PCM (SURVEY Appendix B.1 recipe family: sinusoid mixture + coloured noise + transients)
# ----------------------------------------------------------------------------------------------
def synth_channel(n, sr, seed):
    r = np.random.default_rng(seed)
    t = np.arange(n) / sr
    x = np.zeros(n)
    for f, a in [(220, 0.25), (440, 0.15), (1000 * r.uniform(0.9, 1.1), 0.1), (3300, 0.05)]:
        x += a * np.sin(2 * np.pi * f * t + r.uniform(0, 6.28))
    w = r.standard_normal(n)
    # one-pole-ish colouring: 200-tap exponential FIR, applied by FFT for long signals
    k = 0.95 ** np.arange(200)
    if n > 1 << 16:
        L = 1 << int(np.ceil(np.log2(n + 200)))
        x += np.fft.irfft(np.fft.rfft(w, L) * np.fft.rfft(k, L), L)[:n] * 0.01
    else:
        x += np.convolve(w, k)[:n] * 0.01
    num_tr = max(1, int(round(20 * n / (sr * 10))))
    if n > 2000:
        for p in r.integers(0, n - 2000, size=num_tr):
            x[p:p + 2000] += 0.3 * np.exp(-np.arange(2000) / 200.0) * r.standard_normal(2000)
    return x


def synth_pcm(seconds=10.0, sr=44100, channels=2, bits=16, seed=1, n=None):
    """int32 [C][n] right-justified PCM.  channels=2, bits=16, seconds=10, seed=1 reproduces the
    SURVEY B.1 clip exactly (R = 0.7 L + 0.3 other)."""
    if n is None:
        n = int(round(seconds * sr))
    base = synth_channel(n, sr, seed)
    chans = [base]
    for c in range(1, channels):
        chans.append(0.7 * base + 0.3 * synth_channel(n, sr, seed + c))
    scale = 20000.0 * (1 << (bits - 16)) if bits >= 16 else 20000.0 / (1 << (16 - bits))
    lo, hi = -(1 << (bits - 1)), (1 << (bits - 1)) - 1
    return np.clip(np.round(np.stack(chans, 0) * scale), lo, hi).astype(np.int32)


def reference_test_generators():
    """The nine waveform generators of the reference's round-trip test
    (test/linne_encode_decode/main.cpp:47-188), as float arrays in [-1, 1]."""
    def silence(c, n): return np.zeros((c, n))
    def sine(c, n): return np.tile(np.sin(440.0 * 2 * np.pi * np.arange(n) / 44100.0), (c, 1))
    def sine_flip(c, n): return np.stack([(-1.0) ** ch * np.sin(440.0 * 2 * np.pi * np.arange(n) / 44100.0) for ch in range(c)])
    def white(c, n): return np.random.default_rng(0).uniform(-1.0, 1.0, size=(c, n))
    def chirp(c, n):
        s = np.arange(n); return np.tile(np.sin((2.0 * np.pi * s) / (n - s)), (c, 1))
    def pos(c, n): return np.ones((c, n))
    def neg(c, n): return -np.ones((c, n))
    def nyquist(c, n): return np.tile(np.where(np.arange(n) % 2 == 0, 1.0, -1.0), (c, 1))
    def gauss(c, n): return np.clip(0.25 * np.random.default_rng(1).standard_normal((c, n)), -1.0, 1.0)
    return {"silence": silence, "sine": sine, "sine_flip": sine_flip, "white": white, "chirp": chirp,
            "pos_const": pos, "neg_const": neg, "nyquist": nyquist, "gauss": gauss}


def to_fixed(x, bits):
    """test/linne_encode_decode/main.cpp:191-214: round half away from zero, clip the top."""
    v = np.where(x >= 0, np.floor(x * (1 << (bits - 1)) + 0.5), -np.floor(-x * (1 << (bits - 1)) + 0.5))
    return np.minimum(v, (1 << (bits - 1)) - 1).astype(np.int32)


def mixed_types_pcm(sr=44100, bits=16):
    """3 s stereo: full-scale white noise / digital silence / 440 Hz sine -> RAW, SILENT and
    compressed blocks in one stream (SURVEY Appendix B)."""
    r = np.random.default_rng(7)
    full = (1 << (bits - 1)) - 1
    a = r.integers(-full - 1, full + 1, size=(2, sr))
    b = np.zeros((2, sr), dtype=np.int64)
    c = np.tile(np.round(0.5 * full * np.sin(2 * np.pi * 440 * np.arange(sr) / sr)), (2, 1))
    return np.concatenate([a, b, c], axis=1).astype(np.int32)


def tile_stream(stream: bytes, times: int, block: int) -> bytes:
    """Repeat the full-size blocks of a stream `times` times behind one patched header (legal because
    blocks are self-contained, SURVEY Appendix B 'Block tiling verified')."""
    nch = int.from_bytes(stream[12:14], "big")
    off = 30
    spans = []
    while off < len(stream):
        size = int.from_bytes(stream[off + 2:off + 6], "big") + 6
        ns = int.from_bytes(stream[off + 9:off + 11], "big")
        if ns == block:
            spans.append((off, off + size))
        off += size
    body = b"".join(stream[a:b] for a, b in spans)
    total = len(spans) * block * times
    hdr = bytearray(stream[:30])
    hdr[14:18] = total.to_bytes(4, "big")
    return bytes(hdr) + body * times


# ----------------------------------------------------------------------------------------------
# Host simulator: the product's host C code + kernel bodies compiled for the CPU (tests/hostsim).
# TEST INFRASTRUCTURE for the CPU-only suite; the linne_b200 package never loads it.
# ----------------------------------------------------------------------------------------------
HOSTSIM_SO = os.path.join(ROOT, "tests", "hostsim", "liblinne_hostsim.so")


def have_hostsim() -> bool:
    return os.path.exists(HOSTSIM_SO)


class HostSim(LinneApi):
    def __init__(self):
        from linne_b200.api import bind_ext_api, Product
        super().__init__(bind_ext_api(C.CDLL(HOSTSIM_SO, mode=getattr(os, "RTLD_LOCAL", 0))))
        assert self.lib.LINNEB200_Backend() == b"hostsim"
        self.encode_with_params = Product.encode_with_params.__get__(self)
        self.encode_packed = Product.encode_packed.__get__(self)
        self.decode_packed = Product.decode_packed.__get__(self)


def pack_pcm(pcm, bits):
    """int32 [C][n] right-justified -> interleaved little-endian bytes as in a WAV data chunk."""
    inter = np.ascontiguousarray(pcm.T).reshape(-1).astype(np.int64)
    if bits == 8:
        return ((inter + 128) & 0xFF).astype(np.uint8).tobytes()
    nbytes = bits // 8
    raw = (inter & ((1 << bits) - 1)).astype("<u8").view(np.uint8).reshape(-1, 8)[:, :nbytes]
    return np.ascontiguousarray(raw).tobytes()


def params_from_golden(g):
    """ChannelParams array (block-major) from a tests/golden fixture."""
    from linne_b200.api import ChannelParams
    nb, nch = g["units"].shape[:2]
    arr = (ChannelParams * (nb * nch))()
    for b in range(nb):
        for c in range(nch):
            p = arr[b * nch + c]
            for l in range(3):
                u = int(g["units"][b, c, l])
                p.log2_units[l] = max(u, 1).bit_length() - 1
                p.rshift[l] = int(g["rshift"][b, c, l])
                for i in range(128):
                    p.coef[l][i] = int(g["coef"][b, c, l, i])
    return arr


def load_golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))


GOLDEN_CASES = ["stereo16_m0", "stereo16_m4", "stereo16_m7", "mono8_m7", "eightch24_m7", "mono24_m2"]
