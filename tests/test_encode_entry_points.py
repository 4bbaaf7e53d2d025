"""Every encoder entry point against a literal table of result codes.

A call that succeeds must write what the same backend's plain single-range LINNEEncoder_EncodeWhole writes for the same
PCM (for the corpus calls: every file what its own single-file call writes).  That holds however the call is cut: over
several block ranges (LINNE_B200_GPUS, LINNE_B200_PIPELINE), into several scratch chunks (LINNE_B200_SCRATCH_MB) or
into one batch of several files.  A call given an output buffer of exactly the size it needs, one byte less, or less
than the stream header leaves the buffer (sentinel-filled, with guard bytes behind it) as the table's SHA-256 says: a
refused call writes no more than it did when the table was recorded, and never past the size it was given.

CPU: the host code on the simulator (its "device" memory is host memory).  GPU: the product, resident buffers in HBM."""
import ctypes as C
import hashlib
import os
from contextlib import contextmanager

import numpy as np
import pytest

import harness
from harness import (OK, INVALID_ARGUMENT, INVALID_FORMAT, INSUFFICIENT_BUFFER, PARAMETER_NOT_SET, LINNEEncodeParameter,
                     LINNEEncoderConfig)
from linne_b200.api import ChannelParams, FileDesc, _chan_ptrs

u8p = C.POINTER(C.c_uint8)
SENTINEL, GUARD = 0xA5, 64

# name: channels, bits, block, samples, preset
SIGNALS = {
    "stereo16": (2, 16, 1024, 1024 * 7 + 300, 1),        # 8 blocks with a tail: enough for three block ranges
    "mono8": (1, 8, 1024, 1024 * 2 + 5, 2),
    "eight24": (8, 24, 1024, 1024 * 6 + 100, 0),
    "short": (2, 16, 2048, 500, 3),                      # shorter than one block
    "flat": (1, 16, 16384, 16384 + 3000, 0),             # 16384-sample blocks: the flat analysis kernels on the GPU
    # loud noise: the block type comes from an estimate, and these streams come out longer than their all-raw form
    "noise8": (1, 8, 1024, 4096, 0),
    "noise16": (2, 16, 1024, 8192, 3),
}
ENVS = {
    "plain": {},
    "gpus3": {"LINNE_B200_GPUS": "3"},                   # three block ranges (sharing one device where there is one)
    "pipe2": {"LINNE_B200_PIPELINE": "2"},               # two pipelined ranges on the handle's device
    "scratch1": {"LINNE_B200_SCRATCH_MB": "1"},          # a few blocks per scratch chunk
}

H = {"hostsim": None, "gpu": None}   # no hash: an "ample" call is checked against the plain call's bytes instead

# (entry point, signal, environment, output buffer, result code, SHA-256 of the buffer after the call per backend)
# output buffer: "ample", or the size the plain call needed ("exact"), one byte less ("short"), 29 bytes ("tiny")
ENTRY_TABLE = [
    ("Whole", "stereo16", "plain", "ample", OK, H),
    ("Whole", "mono8", "plain", "ample", OK, H),
    ("Whole", "eight24", "plain", "ample", OK, H),
    ("Whole", "short", "plain", "ample", OK, H),
    ("Whole", "flat", "plain", "ample", OK, H),
    ("Block", "stereo16", "plain", "ample", OK, H),
    ("Block", "mono8", "plain", "ample", OK, H),
    ("Block", "eight24", "plain", "ample", OK, H),
    ("Block", "short", "plain", "ample", OK, H),
    ("Block", "flat", "plain", "ample", OK, H),
    ("WithParams", "stereo16", "plain", "ample", OK, H),
    ("WithParams", "mono8", "plain", "ample", OK, H),
    ("WithParams", "eight24", "plain", "ample", OK, H),
    ("WithParams", "short", "plain", "ample", OK, H),
    ("WithParams", "flat", "plain", "ample", OK, H),
    ("Resident", "stereo16", "plain", "ample", OK, H),
    ("Resident", "mono8", "plain", "ample", OK, H),
    ("Resident", "eight24", "plain", "ample", OK, H),
    ("Resident", "short", "plain", "ample", OK, H),
    ("Resident", "flat", "plain", "ample", OK, H),
    ("Packed", "stereo16", "plain", "ample", OK, H),
    ("Packed", "mono8", "plain", "ample", OK, H),
    ("Packed", "eight24", "plain", "ample", OK, H),
    ("Packed", "short", "plain", "ample", OK, H),
    ("Packed", "flat", "plain", "ample", OK, H),
    ("FilesResident", "stereo16", "plain", "ample", OK, H),
    ("FilesResident", "mono8", "plain", "ample", OK, H),
    ("FilesResident", "eight24", "plain", "ample", OK, H),
    ("FilesResident", "short", "plain", "ample", OK, H),
    ("FilesResident", "flat", "plain", "ample", OK, H),
    ("FilesPacked", "stereo16", "plain", "ample", OK, H),
    ("FilesPacked", "mono8", "plain", "ample", OK, H),
    ("FilesPacked", "eight24", "plain", "ample", OK, H),
    ("FilesPacked", "short", "plain", "ample", OK, H),
    ("FilesPacked", "flat", "plain", "ample", OK, H),
    ("Whole", "stereo16", "gpus3", "ample", OK, H),
    ("Whole", "eight24", "gpus3", "ample", OK, H),
    ("Packed", "stereo16", "gpus3", "ample", OK, H),
    ("Packed", "eight24", "gpus3", "ample", OK, H),
    ("Whole", "stereo16", "pipe2", "ample", OK, H),
    ("Whole", "eight24", "pipe2", "ample", OK, H),
    ("Packed", "stereo16", "pipe2", "ample", OK, H),
    ("Packed", "eight24", "pipe2", "ample", OK, H),
    ("Whole", "stereo16", "scratch1", "ample", OK, H),
    ("Whole", "eight24", "scratch1", "ample", OK, H),
    ("Whole", "flat", "scratch1", "ample", OK, H),
    ("Block", "stereo16", "scratch1", "ample", OK, H),
    ("Block", "flat", "scratch1", "ample", OK, H),
    ("WithParams", "stereo16", "scratch1", "ample", OK, H),
    ("WithParams", "eight24", "scratch1", "ample", OK, H),
    ("WithParams", "flat", "scratch1", "ample", OK, H),
    ("Resident", "stereo16", "scratch1", "ample", OK, H),
    ("Resident", "eight24", "scratch1", "ample", OK, H),
    ("Resident", "flat", "scratch1", "ample", OK, H),
    ("Packed", "stereo16", "scratch1", "ample", OK, H),
    ("Packed", "eight24", "scratch1", "ample", OK, H),
    ("Packed", "flat", "scratch1", "ample", OK, H),
    ("FilesResident", "stereo16", "scratch1", "ample", OK, H),
    ("FilesResident", "eight24", "scratch1", "ample", OK, H),
    ("FilesResident", "flat", "scratch1", "ample", OK, H),
    ("FilesPacked", "stereo16", "scratch1", "ample", OK, H),
    ("FilesPacked", "eight24", "scratch1", "ample", OK, H),
    ("FilesPacked", "flat", "scratch1", "ample", OK, H),
    ("Whole", "noise8", "plain", "ample", OK, H),
    ("Block", "noise8", "plain", "ample", OK, H),
    ("WithParams", "noise8", "plain", "ample", OK, H),
    ("Resident", "noise8", "plain", "ample", OK, H),
    ("Packed", "noise8", "plain", "ample", OK, H),
    ("FilesResident", "noise8", "plain", "ample", OK, H),
    ("FilesPacked", "noise8", "plain", "ample", OK, H),
    ("Whole", "noise16", "plain", "ample", OK, H),
    ("Block", "noise16", "plain", "ample", OK, H),
    ("WithParams", "noise16", "plain", "ample", OK, H),
    ("Resident", "noise16", "plain", "ample", OK, H),
    ("Packed", "noise16", "plain", "ample", OK, H),
    ("FilesResident", "noise16", "plain", "ample", OK, H),
    ("FilesPacked", "noise16", "plain", "ample", OK, H),
    # block ranges of loud noise: longer than their all-raw form, which is what a range used to be given
    ("Whole", "noise16", "gpus3", "ample", OK, H),
    ("Packed", "noise16", "gpus3", "ample", OK, H),
    ("Whole", "noise16", "pipe2", "ample", OK, H),
    ("Packed", "noise16", "pipe2", "ample", OK, H),
    ("Whole", "noise16", "scratch1", "ample", OK, H),
    ("FilesResident", "noise16", "scratch1", "ample", OK, H),
    ("FilesPacked", "noise16", "scratch1", "ample", OK, H),
    ("Whole", "stereo16", "plain", "exact", OK, {"hostsim": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af", "gpu": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af"}),
    ("Whole", "stereo16", "plain", "short", INSUFFICIENT_BUFFER, {"hostsim": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415", "gpu": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415"}),
    ("Whole", "stereo16", "plain", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("Packed", "stereo16", "plain", "exact", OK, {"hostsim": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af", "gpu": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af"}),
    ("Packed", "stereo16", "plain", "short", INSUFFICIENT_BUFFER, {"hostsim": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415", "gpu": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415"}),
    ("Packed", "stereo16", "plain", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("Resident", "stereo16", "plain", "exact", OK, {"hostsim": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af", "gpu": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af"}),
    ("Resident", "stereo16", "plain", "short", INSUFFICIENT_BUFFER, {"hostsim": "77540a1121882611d42d6a59ee5aab53091a2c31aae023987cc83dc752c418f1", "gpu": "77540a1121882611d42d6a59ee5aab53091a2c31aae023987cc83dc752c418f1"}),
    ("Resident", "stereo16", "plain", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("FilesResident", "stereo16", "plain", "exact", OK, {"hostsim": "f06df8961b4fa286ded601c9ebb4cae78dde55ed55b1b1d8352839b78e95193b", "gpu": "f06df8961b4fa286ded601c9ebb4cae78dde55ed55b1b1d8352839b78e95193b"}),
    ("FilesResident", "stereo16", "plain", "short", INSUFFICIENT_BUFFER, {"hostsim": "5880ce682e9af34383dbc35a10ebbb1ddbb13163092c86851fdcc9127447344c", "gpu": "5880ce682e9af34383dbc35a10ebbb1ddbb13163092c86851fdcc9127447344c"}),
    ("FilesResident", "stereo16", "plain", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("FilesPacked", "stereo16", "plain", "exact", OK, {"hostsim": "f06df8961b4fa286ded601c9ebb4cae78dde55ed55b1b1d8352839b78e95193b", "gpu": "f06df8961b4fa286ded601c9ebb4cae78dde55ed55b1b1d8352839b78e95193b"}),
    ("FilesPacked", "stereo16", "plain", "short", INSUFFICIENT_BUFFER, {"hostsim": "65d9562a7240e02d72cc000216fa2f114634cb367b11ed9443503938388603ee", "gpu": "65d9562a7240e02d72cc000216fa2f114634cb367b11ed9443503938388603ee"}),
    ("FilesPacked", "stereo16", "plain", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("Whole", "stereo16", "scratch1", "exact", OK, {"hostsim": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af", "gpu": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af"}),
    ("Whole", "stereo16", "scratch1", "short", INSUFFICIENT_BUFFER, {"hostsim": "7cc1d9c9825c5c765ff9b4aa8df9f8701b818a01f59e725b6eae9564db5742fd", "gpu": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415"}),
    ("Whole", "stereo16", "scratch1", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("Packed", "stereo16", "scratch1", "exact", OK, {"hostsim": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af", "gpu": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af"}),
    ("Packed", "stereo16", "scratch1", "short", INSUFFICIENT_BUFFER, {"hostsim": "7cc1d9c9825c5c765ff9b4aa8df9f8701b818a01f59e725b6eae9564db5742fd", "gpu": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415"}),
    ("Packed", "stereo16", "scratch1", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("Resident", "stereo16", "scratch1", "exact", OK, {"hostsim": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af", "gpu": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af"}),
    ("Resident", "stereo16", "scratch1", "short", INSUFFICIENT_BUFFER, {"hostsim": "77540a1121882611d42d6a59ee5aab53091a2c31aae023987cc83dc752c418f1", "gpu": "77540a1121882611d42d6a59ee5aab53091a2c31aae023987cc83dc752c418f1"}),
    ("Resident", "stereo16", "scratch1", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("FilesResident", "stereo16", "scratch1", "exact", OK, {"hostsim": "f06df8961b4fa286ded601c9ebb4cae78dde55ed55b1b1d8352839b78e95193b", "gpu": "f06df8961b4fa286ded601c9ebb4cae78dde55ed55b1b1d8352839b78e95193b"}),
    ("FilesResident", "stereo16", "scratch1", "short", INSUFFICIENT_BUFFER, {"hostsim": "3465de148fd7e48b85146655fb0d4afc29e3d343ef208a4a0434b188f5c103ba", "gpu": "5880ce682e9af34383dbc35a10ebbb1ddbb13163092c86851fdcc9127447344c"}),
    ("FilesResident", "stereo16", "scratch1", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("FilesPacked", "stereo16", "scratch1", "exact", OK, {"hostsim": "f06df8961b4fa286ded601c9ebb4cae78dde55ed55b1b1d8352839b78e95193b", "gpu": "f06df8961b4fa286ded601c9ebb4cae78dde55ed55b1b1d8352839b78e95193b"}),
    ("FilesPacked", "stereo16", "scratch1", "short", INSUFFICIENT_BUFFER, {"hostsim": "65d9562a7240e02d72cc000216fa2f114634cb367b11ed9443503938388603ee", "gpu": "65d9562a7240e02d72cc000216fa2f114634cb367b11ed9443503938388603ee"}),
    ("FilesPacked", "stereo16", "scratch1", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("Whole", "stereo16", "gpus3", "exact", OK, {"hostsim": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af", "gpu": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af"}),
    ("Whole", "stereo16", "gpus3", "short", INSUFFICIENT_BUFFER, {"hostsim": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415", "gpu": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415"}),
    ("Whole", "stereo16", "gpus3", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
    ("Packed", "stereo16", "gpus3", "exact", OK, {"hostsim": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af", "gpu": "2ad3fc67a0a44287b5ddd3e89e166c2e41880ab6dd5bd096e6f4f73a7902a3af"}),
    ("Packed", "stereo16", "gpus3", "short", INSUFFICIENT_BUFFER, {"hostsim": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415", "gpu": "1fd70642421ccca54798dff68af40040ef17a3a1e6e89fc38170dee481373415"}),
    ("Packed", "stereo16", "gpus3", "tiny", INSUFFICIENT_BUFFER, {"hostsim": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49", "gpu": "41802bce980af3cfc4af88000100a1b5e4e444a2b6936330b4d8b45a0adeec49"}),
]


@contextmanager
def environment(values):
    """exactly `values` of the encoder's environment switches set while inside"""
    names = {n for e in ENVS.values() for n in e}
    old = {n: os.environ.get(n) for n in names}
    for n in names:
        os.environ.pop(n, None)
    os.environ.update(values)
    try:
        yield
    finally:
        for n, v in old.items():
            if v is None:
                os.environ.pop(n, None)
            else:
                os.environ[n] = v


class HostMem:
    """`device` memory of the simulator = host memory"""
    def __init__(self, arr): self.arr = np.ascontiguousarray(arr)
    @property
    def ptr(self): return self.arr.ctypes.data
    def get(self): return self.arr.tobytes()


class CudaMem:
    def __init__(self, arr):
        import torch
        self.t = torch.from_numpy(np.ascontiguousarray(arr)).cuda()
    @property
    def ptr(self): return self.t.data_ptr()
    def get(self):
        import torch
        torch.cuda.synchronize()                         # copies a refused call left in flight on the library's stream
        return self.t.cpu().numpy().tobytes()


class Backend:
    def __init__(self, name, codec, mem):
        self.name, self.codec, self.lib, self.Mem = name, codec, codec.lib, mem
        self.oracle = harness.Oracle()
        self.plain = {}


def signal_pcm(sig):
    ch, bits, _, n, _ = SIGNALS[sig]
    if sig.startswith("noise"):
        full = 1 << (bits - 1)
        noise = np.random.default_rng(7).standard_normal((ch, n)) * 0.4 * full
        return np.clip(np.round(noise), -full, full - 1).astype(np.int32)
    return harness.synth_pcm(n=n, channels=ch, bits=bits, seed=400 + n % 97)


def signal_files(sig):
    """the signal cut into three files"""
    pcm = signal_pcm(sig)
    n = pcm.shape[1]
    if sig.startswith("noise"):                          # whole blocks: nothing of the raw size goes to padding
        a, b = n // 2, n * 3 // 4
    else:
        a = n // 2 + 13
        b = a + (n - a) // 3
    return [np.ascontiguousarray(pcm[:, lo:hi]) for lo, hi in ((0, a), (a, b), (b, n))]


def ample(pcm):
    return 30 + 2 * pcm.size * 4 + 4096


def make_encoder(L, sig, configure=True, bits=None):
    ch, sbits, block, _, preset = SIGNALS[sig]
    enc = L.LINNEEncoder_Create(C.byref(LINNEEncoderConfig(ch, block, 3, 128)), None, 0)
    assert enc
    if configure:
        prm = LINNEEncodeParameter(ch, bits or sbits, 44100, block, preset, 1 if ch >= 2 else 0, 0, 0)
        assert L.LINNEEncoder_SetEncodeParameter(enc, C.byref(prm)) == OK
    return enc


def sentinel(size):
    return np.full(size + GUARD, SENTINEL, np.uint8)


def zero_params(sig):
    ch, _, block, n, _ = SIGNALS[sig]
    return (ChannelParams * (-(-n // block) * ch))()


# ---- one call of each entry point: (result code, the streams it wrote, the whole output buffer afterwards) ----------
def call_whole(be, enc, sig, cap):
    pcm = signal_pcm(sig)
    out, size = sentinel(cap), C.c_uint32(0)
    rc = be.lib.LINNEEncoder_EncodeWhole(enc, _chan_ptrs(pcm), pcm.shape[1], out.ctypes.data_as(u8p), cap, C.byref(size))
    return rc, [out[:size.value].tobytes()], out.tobytes()


def call_block(be, enc, sig, cap):
    """the command-line tool's loop: the header, then one LINNEEncoder_EncodeBlock per block"""
    ch, bits, block, n, preset = SIGNALS[sig]
    pcm = signal_pcm(sig)
    out = sentinel(cap)
    hdr = harness.LINNEHeader(1, 2, ch, n, 44100, bits, block, preset, 1 if ch >= 2 else 0)
    rc = be.lib.LINNEEncoder_EncodeHeader(C.byref(hdr), out.ctypes.data_as(u8p), cap)
    off, done, size = 30, 0, C.c_uint32(0)
    while rc == OK and done < n:
        m = min(block, n - done)
        sub = (C.POINTER(C.c_int32) * ch)(*[C.cast(pcm[c].ctypes.data + 4 * done, C.POINTER(C.c_int32)) for c in range(ch)])
        rc = be.lib.LINNEEncoder_EncodeBlock(enc, sub, m, C.cast(out.ctypes.data + off, u8p), cap - off, C.byref(size))
        off, done = off + size.value, done + m
    return rc, [out[:off].tobytes()], out.tobytes()


def call_with_params(be, enc, sig, cap):
    pcm = signal_pcm(sig)
    params = zero_params(sig)
    out, size = sentinel(cap), C.c_uint32(0)
    rc = be.lib.LINNEB200_EncodeWholeWithParams(enc, _chan_ptrs(pcm), pcm.shape[1], params, len(params) // pcm.shape[0],
                                                out.ctypes.data_as(u8p), cap, C.byref(size))
    return rc, [out[:size.value].tobytes()], out.tobytes()


def call_resident(be, enc, sig, cap):
    pcm = signal_pcm(sig)
    stride = pcm.shape[1] + 5
    planes = np.zeros((pcm.shape[0], stride), np.int32)
    planes[:, :pcm.shape[1]] = pcm
    d_pcm, d_out, size = be.Mem(planes), be.Mem(sentinel(cap)), C.c_uint32(0)
    rc = be.lib.LINNEB200_EncodeWholeResident(enc, C.c_void_p(d_pcm.ptr), stride, pcm.shape[1], C.c_void_p(d_out.ptr), cap,
                                              C.byref(size))
    buf = d_out.get()
    return rc, [buf[:size.value]], buf


def call_packed(be, enc, sig, cap):
    pcm = signal_pcm(sig)
    src = np.frombuffer(harness.pack_pcm(pcm, SIGNALS[sig][1]), np.uint8).copy()
    out, size = sentinel(cap), C.c_uint32(0)
    rc = be.lib.LINNEB200_EncodeWholePacked(enc, src.ctypes.data_as(u8p), pcm.shape[1], out.ctypes.data_as(u8p), cap, C.byref(size))
    return rc, [out[:size.value].tobytes()], out.tobytes()


def files_streams(buf, desc):
    return [buf[d.out_offset:d.out_offset + d.out_size] for d in desc]


def call_files_resident(be, enc, sig, cap):
    files = signal_files(sig)
    starts, off = [], 16                                 # files need not start at sample 0 nor touch each other
    for f in files:
        starts.append(off); off += f.shape[1] + 24
    planes = np.zeros((files[0].shape[0], off), np.int32)
    for f, s in zip(files, starts):
        planes[:, s:s + f.shape[1]] = f
    desc = (FileDesc * len(files))(*[FileDesc(s, f.shape[1], 0, 0, 0) for f, s in zip(files, starts)])
    d_pcm, d_out, size = be.Mem(planes), be.Mem(sentinel(cap)), C.c_uint32(0)
    rc = be.lib.LINNEB200_EncodeFilesResident(enc, C.c_void_p(d_pcm.ptr), off, desc, len(files), C.c_void_p(d_out.ptr), cap,
                                              C.byref(size))
    buf = d_out.get()
    return rc, files_streams(buf, desc) if rc == OK else [], buf


def call_files_packed(be, enc, sig, cap):
    files = signal_files(sig)
    src = np.frombuffer(b"".join(harness.pack_pcm(f, SIGNALS[sig][1]) for f in files), np.uint8).copy()
    desc = (FileDesc * len(files))(*[FileDesc(0, f.shape[1], 0, 0, 0) for f in files])
    out, size = sentinel(cap), C.c_uint32(0)
    rc = be.lib.LINNEB200_EncodeFilesPacked(enc, src.ctypes.data_as(u8p), desc, len(files), out.ctypes.data_as(u8p), cap, C.byref(size))
    return rc, files_streams(out.tobytes(), desc) if rc == OK else [], out.tobytes()


CALLS = {"Whole": call_whole, "Block": call_block, "WithParams": call_with_params, "Resident": call_resident,
         "Packed": call_packed, "FilesResident": call_files_resident, "FilesPacked": call_files_packed}


def run(be, kind, sig, env, cap=None):
    if cap is None:
        cap = ample(signal_pcm(sig))
    with environment(ENVS[env]):
        enc = make_encoder(be.lib, sig)
        try:
            return CALLS[kind](be, enc, sig, cap)
        finally:
            be.lib.LINNEEncoder_Destroy(enc)


def plain(be, kind, sig):
    """what the call must write: the plain single-range EncodeWhole of the same PCM, of each file for the corpus calls
    (WithParams: the plain single-range call with the same parameters)"""
    key = {"WithParams": "WithParams", "FilesResident": "Files", "FilesPacked": "Files"}.get(kind, "Whole"), sig
    if key not in be.plain:
        ch, bits, block, _, preset = SIGNALS[sig]
        with environment({}):
            if key[0] == "WithParams":
                be.plain[key] = run(be, "WithParams", sig, "plain")[1]
            else:
                pcms = signal_files(sig) if key[0] == "Files" else [signal_pcm(sig)]
                be.plain[key] = [be.codec.encode(p, bits=bits, preset=preset, block=block) for p in pcms]
    return be.plain[key]


def observe(be, row):
    """-> (result code, SHA-256 of the output buffer or None) of one table row; the streams of an OK call are checked"""
    kind, sig, env, buf = row[:4]
    want = plain(be, kind, sig)
    need = sum(len(s) for s in want)
    cap = {"ample": None, "exact": need, "short": need - 1, "tiny": 29}[buf]
    rc, streams, image = run(be, kind, sig, env, cap)
    if rc == OK:
        assert streams == want, "differs from the plain single-range call"
        pcms = signal_files(sig) if kind.startswith("Files") else [signal_pcm(sig)]
        assert all(np.array_equal(be.oracle.decode(s), p) for s, p in zip(streams, pcms)), "the oracle does not decode it back"
    return rc, None if buf == "ample" else hashlib.sha256(image).hexdigest()


def check_row(be, row):
    rc, digest = observe(be, row)
    assert rc == row[4]
    assert digest == row[5][be.name]


def row_id(row):
    return "-".join(row[:4])


@pytest.fixture(scope="module")
def hostsim_backend(hostsim):
    return Backend("hostsim", hostsim, HostMem)


@pytest.fixture(scope="module")
def gpu_backend(gpu):
    return Backend("gpu", gpu, CudaMem)


@pytest.mark.parametrize("row", ENTRY_TABLE, ids=row_id)
def test_entry_point_hostsim(hostsim_backend, row):
    check_row(hostsim_backend, row)


@pytest.mark.gpu
@pytest.mark.parametrize("row", ENTRY_TABLE, ids=row_id)
def test_entry_point_gpu(gpu_backend, row):
    check_row(gpu_backend, row)


# ---- rejections ---------------------------------------------------------------------------------------------------
def reject_not_set(kind):
    def call(be):
        enc = make_encoder(be.lib, "stereo16", configure=False)
        try:
            return CALLS[kind](be, enc, "stereo16", ample(signal_pcm("stereo16")))[0]
        finally:
            be.lib.LINNEEncoder_Destroy(enc)
    return call


def with_encoder(body, sig="stereo16", env="plain", bits=None):
    def call(be):
        with environment(ENVS[env]):
            enc = make_encoder(be.lib, sig, bits=bits)
            try:
                return body(be, enc)
            finally:
                be.lib.LINNEEncoder_Destroy(enc)
    return call


def null_plane(kind):
    def body(be, enc):
        pcm = signal_pcm("stereo16")
        ptrs = _chan_ptrs(pcm)
        ptrs[1] = C.POINTER(C.c_int32)()
        out, size = sentinel(ample(pcm)), C.c_uint32(0)
        if kind == "Block":
            return be.lib.LINNEEncoder_EncodeBlock(enc, ptrs, 1024, out.ctypes.data_as(u8p), len(out), C.byref(size))
        if kind == "WithParams":
            params = zero_params("stereo16")
            return be.lib.LINNEB200_EncodeWholeWithParams(enc, ptrs, pcm.shape[1], params, len(params) // 2,
                                                          out.ctypes.data_as(u8p), len(out), C.byref(size))
        return be.lib.LINNEEncoder_EncodeWhole(enc, ptrs, pcm.shape[1], out.ctypes.data_as(u8p), len(out), C.byref(size))
    return body


def bad_params(field, value):
    def body(be, enc):
        params = zero_params("stereo16")
        getattr(params[5], field)[1] = value
        return call_params(be, enc, params, signal_pcm("stereo16").shape[1], len(params) // 2)
    return body


def call_params(be, enc, params, n, num_param_blocks):
    pcm = signal_pcm("stereo16")
    out, size = sentinel(ample(pcm)), C.c_uint32(0)
    return be.lib.LINNEB200_EncodeWholeWithParams(enc, _chan_ptrs(pcm), n, params, num_param_blocks,
                                                  out.ctypes.data_as(u8p), len(out), C.byref(size))


def params_wrap(be, enc):
    """ceil(n / block) of n = 2^32 - 1 wraps in 32 bits: a block count near 0 would pass for the records given"""
    return call_params(be, enc, zero_params("stereo16"), 0xFFFFFFFF, 0)


def files_call(kind, first, lengths, stride):
    def body(be, enc):
        pcm = signal_pcm("stereo16")
        desc = (FileDesc * len(lengths))(*[FileDesc(first, n, 0, 0, 0) for n in lengths])
        cap = ample(pcm)
        out, size = sentinel(cap), C.c_uint32(0)
        if kind == "FilesPacked":
            src = np.frombuffer(harness.pack_pcm(pcm, 16), np.uint8).copy()
            return be.lib.LINNEB200_EncodeFilesPacked(enc, src.ctypes.data_as(u8p), desc, len(desc), out.ctypes.data_as(u8p),
                                                      cap, C.byref(size))
        d_pcm, d_out = be.Mem(pcm), be.Mem(out)
        return be.lib.LINNEB200_EncodeFilesResident(enc, C.c_void_p(d_pcm.ptr), stride, desc, len(desc), C.c_void_p(d_out.ptr),
                                                    cap, C.byref(size))
    return body


def packed_12_bits(kind):
    def body(be, enc):
        pcm = signal_pcm("stereo16")
        src = np.frombuffer(harness.pack_pcm(pcm, 16), np.uint8).copy()
        cap = ample(pcm)
        out, size = sentinel(cap), C.c_uint32(0)
        if kind == "Packed":
            return be.lib.LINNEB200_EncodeWholePacked(enc, src.ctypes.data_as(u8p), pcm.shape[1], out.ctypes.data_as(u8p),
                                                      cap, C.byref(size))
        desc = (FileDesc * 1)(FileDesc(0, pcm.shape[1], 0, 0, 0))
        return be.lib.LINNEB200_EncodeFilesPacked(enc, src.ctypes.data_as(u8p), desc, 1, out.ctypes.data_as(u8p), cap, C.byref(size))
    return body


def resident_stride(be, enc):
    pcm = signal_pcm("stereo16")
    d_pcm, d_out, size = be.Mem(pcm), be.Mem(sentinel(ample(pcm))), C.c_uint32(0)
    return be.lib.LINNEB200_EncodeWholeResident(enc, C.c_void_p(d_pcm.ptr), pcm.shape[1] - 1, pcm.shape[1],
                                                C.c_void_p(d_out.ptr), ample(pcm), C.byref(size))


def block_samples(n):
    def body(be, enc):
        pcm = signal_pcm("stereo16")
        out, size = sentinel(ample(pcm)), C.c_uint32(0)
        return be.lib.LINNEEncoder_EncodeBlock(enc, _chan_ptrs(pcm), n, out.ctypes.data_as(u8p), len(out), C.byref(size))
    return body


N16 = SIGNALS["stereo16"][3]
REJECTIONS = {
    "not_set-Whole": (reject_not_set("Whole"), PARAMETER_NOT_SET),
    "not_set-Block": (reject_not_set("Block"), PARAMETER_NOT_SET),
    "not_set-WithParams": (reject_not_set("WithParams"), PARAMETER_NOT_SET),
    "not_set-Resident": (reject_not_set("Resident"), PARAMETER_NOT_SET),
    "not_set-Packed": (reject_not_set("Packed"), PARAMETER_NOT_SET),
    "not_set-FilesResident": (reject_not_set("FilesResident"), PARAMETER_NOT_SET),
    "not_set-FilesPacked": (reject_not_set("FilesPacked"), PARAMETER_NOT_SET),
    "null_plane-Whole": (with_encoder(null_plane("Whole")), INVALID_ARGUMENT),
    "null_plane-Whole-gpus3": (with_encoder(null_plane("Whole"), env="gpus3"), INVALID_ARGUMENT),
    "null_plane-Block": (with_encoder(null_plane("Block")), INVALID_ARGUMENT),
    "null_plane-WithParams": (with_encoder(null_plane("WithParams")), INVALID_ARGUMENT),
    "bits12-Packed": (with_encoder(packed_12_bits("Packed"), bits=12), INVALID_FORMAT),
    "bits12-FilesPacked": (with_encoder(packed_12_bits("FilesPacked"), bits=12), INVALID_FORMAT),
    "log2_units8-WithParams": (with_encoder(bad_params("log2_units", 8)), INVALID_ARGUMENT),
    "rshift16-WithParams": (with_encoder(bad_params("rshift", 16)), INVALID_ARGUMENT),
    "few_records-WithParams": (with_encoder(lambda be, enc: call_params(be, enc, zero_params("stereo16"), N16, 7)),
                               INVALID_ARGUMENT),
    "wrapping_block_count-WithParams": (with_encoder(params_wrap), INVALID_ARGUMENT),
    "empty_file-FilesResident": (with_encoder(files_call("FilesResident", 0, [1000, 0], N16)), INVALID_ARGUMENT),
    "empty_file-FilesPacked": (with_encoder(files_call("FilesPacked", 0, [1000, 0], N16)), INVALID_ARGUMENT),
    "past_stride-FilesResident": (with_encoder(files_call("FilesResident", 100, [N16 - 99], N16)), INVALID_ARGUMENT),
    "stride_short-Resident": (with_encoder(resident_stride), INVALID_ARGUMENT),
    "too_long-Block": (with_encoder(block_samples(1025)), INSUFFICIENT_BUFFER),
    "no_samples-Block": (with_encoder(block_samples(0)), INVALID_ARGUMENT),
}


@pytest.mark.parametrize("name", sorted(REJECTIONS))
def test_rejection_hostsim(hostsim_backend, name):
    call, want = REJECTIONS[name]
    assert call(hostsim_backend) == want


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(REJECTIONS))
def test_rejection_gpu(gpu_backend, name):
    call, want = REJECTIONS[name]
    assert call(gpu_backend) == want
