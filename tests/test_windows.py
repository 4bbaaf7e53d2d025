"""Random access: LINNEB200_DecoderBuildIndex (one seek point per block) and LINNEB200_DecodeWindows[Resident] (sample
windows of a stream, the blocks they need decoded as one batch).  Every window must equal the DecodeWhole slice bit for
bit, the output planes outside the windows must keep their sentinel, and stream damage must be confined to the windows
that need the damaged block.

CPU: the host code on the simulator (its "device" memory is host memory).  GPU: the product, buffers in HBM."""
import ctypes as C

import numpy as np
import pytest

import harness
from harness import (OK, INVALID_ARGUMENT, INVALID_FORMAT, INSUFFICIENT_BUFFER, INSUFFICIENT_DATA, PARAMETER_NOT_SET,
                     DATA_CORRUPTION, LINNEDecoderConfig)
from linne_b200.api import SeekPoint, StageStat, Window, index_points
from test_corpus_batches import HostMem, CudaMem

BLOCK = 2048
SENTINEL = -7
u8p = C.POINTER(C.c_uint8)


def u8(a):
    return a.ctypes.data_as(u8p)


class Decoder:
    """one decoder handle of the library under test"""

    def __init__(self, codec, channels, check_crc=1):
        self.L = codec.lib
        self.h = self.L.LINNEDecoder_Create(C.byref(LINNEDecoderConfig(channels, 3, 128, check_crc)), None, 0)
        assert self.h

    def close(self):
        self.L.LINNEDecoder_Destroy(self.h)

    def index(self, data=None, d_data=None, size=None, capacity=None):
        n = C.c_uint32(0)
        host = u8(data) if data is not None else None
        dev = C.c_void_p(d_data.ptr) if d_data is not None else None
        rc = self.L.LINNEB200_DecoderBuildIndex(self.h, host, dev, size, None, 0, C.byref(n))
        cap = n.value if capacity is None else capacity
        pts = (SeekPoint * max(1, cap))()
        rc = self.L.LINNEB200_DecoderBuildIndex(self.h, host, dev, size, pts, cap, C.byref(n))
        got = np.frombuffer(bytes(pts), np.uint32).reshape(-1, 2)[:min(cap, n.value)].copy()
        return rc, got, n.value

    def windows(self, data, size, index, spec, channels, room):
        """host buffers: windows (first, len, out_offset) into [channels][room] planes filled with the sentinel"""
        pts, npts = index_points(index)
        wins = (Window * max(1, len(spec)))(*[Window(s, n, o, 99) for s, n, o in spec])
        out = np.full((channels, room), SENTINEL, np.int32)
        rc = self.L.LINNEB200_DecodeWindows(self.h, u8(data), size, pts, npts, wins, len(spec), harness._chan_ptrs(out), channels, room)
        return rc, out, [wins[i].status for i in range(len(spec))]

    def windows_resident(self, Mem, d_data, size, index, spec, channels, stride):
        pts, npts = index_points(index)
        wins = (Window * max(1, len(spec)))(*[Window(s, n, o, 99) for s, n, o in spec])
        d_out = Mem(np.full((channels, stride), SENTINEL, np.int32))
        rc = self.L.LINNEB200_DecodeWindowsResident(self.h, C.c_void_p(d_data.ptr), size, pts, npts, wins, len(spec),
                                                    C.c_void_p(d_out.ptr), stride)
        return rc, d_out.get(), [wins[i].status for i in range(len(spec))]


def padded(data):
    buf = np.zeros(len(data) + 16, np.uint8)
    buf[:len(data)] = np.frombuffer(data, np.uint8)
    return buf


def layout(spec_windows, gap=5):
    """(first, len) -> (first, len, out_offset): windows side by side with gaps the sentinel must survive in"""
    out, off = [], 3
    for s, n in spec_windows:
        out.append((s, n, off))
        off += n + gap
    return out, off + 1


def expect(full, spec, channels, room, ok=None):
    want = np.full((channels, room), SENTINEL, np.int32)
    for i, (s, n, o) in enumerate(spec):
        if ok is None or ok[i]:
            want[:, o:o + n] = full[:, s:s + n]
    return want


def check_exact(codec, Mem, data, full, spec_windows, index=None):
    """both entry points: every window equals the DecodeWhole slice, nothing else is written"""
    C_, n = full.shape
    spec, room = layout(spec_windows)
    dec = Decoder(codec, C_)
    host = padded(data)
    d_data = Mem(host)
    try:
        rc, idx, _ = dec.index(host, size=len(data))
        assert rc == OK
        if index is not None:
            idx = index
        rc, out, st = dec.windows(host, len(data), idx, spec, C_, room)
        assert rc == OK and st == [OK] * len(spec)
        assert np.array_equal(out, expect(full, spec, C_, room))
        stride = (room + 3) // 4 * 4 + 4
        rc, out, st = dec.windows_resident(Mem, d_data, len(data), idx, spec, C_, stride)
        assert rc == OK and st == [OK] * len(spec)
        assert np.array_equal(out, expect(full, spec, C_, stride))
    finally:
        dec.close()
    return idx


def shapes(n, idx):
    """inside one block, across block boundaries, the whole stream, the last sample, zero length, overlapping,
    duplicate and unsorted windows"""
    b1 = int(idx[1][0]) if len(idx) > 1 else n
    return [(5, 100), (b1 - 10, 30), (0, n), (n - 1, 1), (123, 0), (n // 2, n // 3), (b1 - 10, 30),
            (b1 + 7, 2 * BLOCK + 3), (1, 1), (n - 1000, 1000), (n // 2 + 10, 50), (n, 0)]


def stream_cases():
    return [(2, 16, 0), (1, 24, 5), (8, 24, 3), (2, 8, 7)]


def run_streams(codec, Mem, oracle, channels, bits, preset, ms):
    pcm = harness.synth_pcm(n=BLOCK * 6 + 777, channels=channels, bits=bits, seed=40 + preset + channels)
    data = oracle.encode(pcm, bits=bits, preset=preset, block=BLOCK, ms=ms)
    full = codec.decode(data)
    assert np.array_equal(full, pcm)
    dec = Decoder(codec, channels)
    try:
        _, idx, _ = dec.index(padded(data), size=len(data))
    finally:
        dec.close()
    assert len(idx) == 7 and list(idx[0]) == [0, 30]
    assert [int(s) for s, _ in idx] == [k * BLOCK for k in range(7)]
    check_exact(codec, Mem, data, full, shapes(full.shape[1], idx))


def mixed_types_stream(oracle):
    """compressed, silent and raw blocks (full-scale noise does not compress) and a tail block"""
    rng = np.random.default_rng(9)
    pcm = harness.synth_pcm(n=BLOCK * 5 + 300, channels=2, bits=16, seed=11)
    pcm[:, BLOCK:2 * BLOCK] = 0
    pcm[:, 3 * BLOCK:4 * BLOCK] = rng.integers(-32768, 32768, size=(2, BLOCK), dtype=np.int32)
    return pcm, oracle.encode(pcm, preset=3, block=BLOCK)


def run_block_types(codec, Mem, oracle):
    pcm, data = mixed_types_stream(oracle)
    full = codec.decode(data)
    assert np.array_equal(full, pcm)
    idx = check_exact(codec, Mem, data, full, shapes(full.shape[1], codec.build_index(data)))
    types = {data[int(off) + 8] for _, off in idx}
    assert {0, 1, 2} <= types, types
    # blocks longer than the header's block size
    stream = bytearray(oracle.encode(pcm, preset=5, block=BLOCK))
    stream[24:28] = (1024).to_bytes(4, "big")
    stream = bytes(stream)
    full = codec.decode(stream)
    assert np.array_equal(full, pcm)
    check_exact(codec, Mem, stream, full, shapes(full.shape[1], codec.build_index(stream)))


def run_indexes(codec, Mem, oracle):
    pcm = harness.synth_pcm(n=BLOCK * 7 + 5, channels=2, bits=16, seed=21)
    data = oracle.encode(pcm, preset=2, block=BLOCK)
    host = padded(data)
    d_data = Mem(host)
    dec = Decoder(codec, 2)
    try:
        rc, on_host, n = dec.index(host, size=len(data))
        assert rc == OK and n == 8
        rc, on_dev, n = dec.index(None, d_data, size=len(data))
        assert rc == OK and n == 8
        assert np.array_equal(on_host, on_dev)
        # too small a capacity: the count, and INSUFFICIENT_BUFFER
        rc, some, n = dec.index(host, size=len(data), capacity=3)
        assert rc == INSUFFICIENT_BUFFER and n == 8 and np.array_equal(some, on_host[:3])
        # a player seeks: DecodeBlock from points[k] yields the DecodeWhole samples of block k and the ones after it
        full = codec.decode(data)
        out = np.zeros((2, BLOCK * 2), np.int32)
        for k in (3, 7, 5):
            first, off = int(on_host[k][0]), int(on_host[k][1])
            used, got = C.c_uint32(0), C.c_uint32(0)
            sub = host[off:]
            assert dec.L.LINNEDecoder_DecodeBlock(dec.h, u8(sub), len(data) - off, harness._chan_ptrs(out), 2, out.shape[1],
                                                  C.byref(used), C.byref(got)) == OK
            assert np.array_equal(out[:, :got.value], full[:, first:first + got.value])
            if k + 1 < len(on_host):
                assert used.value == int(on_host[k + 1][1]) - off
        # a damaged stream: the points before the damage, and the hop's result
        bad = bytearray(data)
        bad[int(on_host[4][1])] ^= 0xFF
        rc, part, n = dec.index(padded(bytes(bad)), size=len(bad))
        assert rc == INVALID_FORMAT and n == 4 and np.array_equal(part, on_host[:4])
        rc, part, n = dec.index(None, Mem(padded(bytes(bad))), size=len(bad))
        assert rc == INVALID_FORMAT and n == 4 and np.array_equal(part, on_host[:4])
    finally:
        dec.close()


def run_rejected(codec, Mem, oracle):
    pcm = harness.synth_pcm(n=BLOCK * 4 + 100, channels=2, bits=16, seed=31)
    data = oracle.encode(pcm, preset=1, block=BLOCK)
    n = pcm.shape[1]
    host = padded(data)
    d_data = Mem(host)
    fresh = Decoder(codec, 2)
    dec = Decoder(codec, 2)
    try:
        # no header latched
        idx = codec.build_index(data)
        spec = [(0, 10, 0)]
        rc, out, st = fresh.windows(host, len(data), idx, spec, 2, 16)
        assert rc == PARAMETER_NOT_SET and st == [99] and np.all(out == SENTINEL)
        rc, _, _ = dec.index(host, size=len(data))
        assert rc == OK

        def rejected(index, spec, room=64, channels=2, want=INVALID_ARGUMENT):
            rc, out, st = dec.windows(host, len(data), index, spec, channels, room)
            assert rc == want and st == [99] * len(spec) and np.all(out == SENTINEL), (rc, st)
            if channels == 2:
                rc, out, st = dec.windows_resident(Mem, d_data, len(data), index, spec, 2, room)
                assert rc == want and st == [99] * len(spec) and np.all(out == SENTINEL), (rc, st)

        good = [(0, 10, 0), (n - 10, 10, 20)]
        rejected(idx, good + [(n - 5, 6, 40)])                       # a window past the end
        rejected(idx, good + [(0, 10, 60)])                          # an output range outside the buffer
        rejected(idx, good, room=25)
        bad = idx.copy(); bad[[1, 2]] = bad[[2, 1]]                  # not monotone
        rejected(bad, good)
        bad = idx.copy(); bad[2][1] = bad[1][1]                      # not strictly increasing
        rejected(bad, good)
        bad = idx.copy(); bad[0][1] = 31                             # does not start at (0, 30)
        rejected(bad, good)
        bad = idx.copy(); bad[0][0] = 1
        rejected(bad, good)
        bad = np.vstack([idx, [[n - 1, len(data)]]]).astype(np.uint32)   # a point beyond the image
        rejected(bad, good)
        rejected(idx, good, channels=1, want=INSUFFICIENT_BUFFER)    # too few channels in the buffer
        # what was rejected left the handle usable
        spec, room = layout([(5, 100), (n - 1, 1)])
        rc, out, st = dec.windows(host, len(data), idx, spec, 2, room)
        assert rc == OK and np.array_equal(out, expect(pcm, spec, 2, room))
    finally:
        fresh.close()
        dec.close()


def run_damage(codec, Mem, oracle):
    pcm = harness.synth_pcm(n=BLOCK * 6 + 300, channels=2, bits=16, seed=51)
    data = oracle.encode(pcm, preset=4, block=BLOCK)
    n = pcm.shape[1]
    idx = codec.build_index(data)
    starts = [int(s) for s, _ in idx]
    windows = [(10, 50), (starts[2] + 5, 40), (starts[1] + 100, BLOCK), (starts[3] - 20, 40), (starts[4], 10), (0, n),
               (n - 5, 5), (7, 0)]
    spec, room = layout(windows)
    needs = [set(np.searchsorted(starts, [s, s + ln - 1], side="right") - 1) if ln else set() for s, ln in windows]
    needs = [set(range(min(k), max(k) + 1)) if k else set() for k in needs]

    def run(image, size, index, check_crc=1):
        host = padded(bytes(image[:size]))
        dec = Decoder(codec, 2, check_crc)
        try:
            dec.L.LINNEDecoder_SetHeader(dec.h, C.byref(codec.decode_header(data)[1]))
            a = dec.windows(host, size, index, spec, 2, room)
            stride = (room + 3) // 4 * 4
            b = dec.windows_resident(Mem, Mem(host), size, index, spec, 2, stride)
            return a, b, stride
        finally:
            dec.close()

    def verify(result, bad_block, code):
        (rc, out, st), (rc2, out2, st2), stride = result
        want = [code if bad_block in nd else OK for nd in needs]
        assert st == want and st2 == want, (st, st2, want)
        first = next((s for s in want if s != OK), OK)
        assert rc == first and rc2 == first
        for o, room_ in ((out, room), (out2, stride)):
            ref = expect(pcm, spec, 2, room_)
            for (s, ln, off), w in zip(spec, want):
                if w != OK:
                    ref[:, off:off + ln] = o[:, off:off + ln]        # undefined
            assert np.array_equal(o, ref)

    # a flipped payload byte in block 2: only the windows that touch it
    bad = bytearray(data)
    bad[int(idx[2][1]) + 40] ^= 0x10
    verify(run(bad, len(bad), idx), 2, DATA_CORRUPTION)
    (rc, _, _), (rc2, _, _), _ = run(bad, len(bad), idx, check_crc=0)
    assert rc == OK and rc2 == OK
    # a point moved into the middle of block 3
    moved = idx.copy()
    moved[3][1] += 17
    verify(run(data, len(data), moved), 3, INVALID_FORMAT)
    # a truncated image: the last block runs past it
    cut = int(idx[-1][1]) + 20
    verify(run(data, cut, idx), len(idx) - 1, INSUFFICIENT_DATA)


def run_readahead_interleaved(codec, Mem, oracle):
    """DecodeWindows between DecodeBlock calls of a read-ahead handle changes none of the blocks DecodeBlock returns"""
    pcm = harness.synth_pcm(n=BLOCK * 8 + 50, channels=2, bits=16, seed=61)
    data = oracle.encode(pcm, preset=2, block=BLOCK)
    other = oracle.encode(harness.synth_pcm(n=BLOCK * 3, channels=2, bits=16, seed=62), preset=2, block=BLOCK)
    host, ohost = padded(data), padded(other)
    dec = Decoder(codec, 2)
    try:
        dec.L.LINNEB200_DecoderSetReadahead(dec.h, 4)
        assert dec.L.LINNEDecoder_SetHeader(dec.h, C.byref(codec.decode_header(data)[1])) == OK
        oidx = codec.build_index(other)
        idx = codec.build_index(data)
        out = np.zeros((2, BLOCK), np.int32)
        off, done = 30, 0
        while done < pcm.shape[1]:
            used, got = C.c_uint32(0), C.c_uint32(0)
            assert dec.L.LINNEDecoder_DecodeBlock(dec.h, u8(host[off:]), len(data) - off, harness._chan_ptrs(out), 2, BLOCK,
                                                  C.byref(used), C.byref(got)) == OK
            assert np.array_equal(out[:, :got.value], pcm[:, done:done + got.value])
            off += used.value
            done += got.value
            # windows of this stream and of another one with the same parameters (the header stays this stream's)
            spec, room = layout([(100, 3000), (done // 2, 17)])
            rc, w, _ = dec.windows(host, len(data), idx, spec, 2, room)
            assert rc == OK and np.array_equal(w, expect(pcm, spec, 2, room))
            rc, w, _ = dec.windows_resident(Mem, Mem(ohost), len(other), oidx, [(5, 9, 0)], 2, 16)
            assert rc == OK
        assert done == pcm.shape[1]
    finally:
        dec.close()


# ---- the simulator -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("channels,bits,preset", stream_cases())
@pytest.mark.parametrize("ms", [0, 1])
def test_windows_streams_hostsim(hostsim, oracle, channels, bits, preset, ms):
    if channels == 1 and ms:
        pytest.skip("M/S needs two channels")
    run_streams(hostsim, HostMem, oracle, channels, bits, preset, ms)


def test_windows_block_types_hostsim(hostsim, oracle):
    run_block_types(hostsim, HostMem, oracle)


def test_windows_indexes_hostsim(hostsim, oracle):
    run_indexes(hostsim, HostMem, oracle)


def test_windows_rejected_hostsim(hostsim, oracle):
    run_rejected(hostsim, HostMem, oracle)


def test_windows_damage_hostsim(hostsim, oracle):
    run_damage(hostsim, HostMem, oracle)


def test_windows_readahead_interleaved_hostsim(hostsim, oracle):
    run_readahead_interleaved(hostsim, HostMem, oracle)


def test_decode_windows_python_api_hostsim(hostsim, oracle):
    pcm = harness.synth_pcm(n=BLOCK * 3 + 10, channels=2, bits=16, seed=71)
    data = oracle.encode(pcm, preset=0, block=BLOCK)
    idx = hostsim.build_index(data)
    assert idx.dtype == np.uint32 and idx.shape == (4, 2)
    for index in (None, idx):
        got = hostsim.decode_windows(data, [3, BLOCK - 1, 0], [10, 5, 0], index=index)
        assert [g.shape for g in got] == [(2, 10), (2, 5), (2, 0)]
        assert np.array_equal(got[0], pcm[:, 3:13]) and np.array_equal(got[1], pcm[:, BLOCK - 1:BLOCK + 4])
    rc, got, st = hostsim.decode_windows(data, [0, len(pcm[0]) - 1], [5, 2], return_code=True)
    assert rc == INVALID_ARGUMENT and st == [0, 0]


# ---- the product ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("channels,bits,preset", stream_cases())
@pytest.mark.parametrize("ms", [0, 1])
def test_windows_streams_gpu(gpu, oracle, channels, bits, preset, ms):
    if channels == 1 and ms:
        pytest.skip("M/S needs two channels")
    run_streams(gpu, CudaMem, oracle, channels, bits, preset, ms)


@pytest.mark.gpu
def test_windows_block_types_gpu(gpu, oracle):
    run_block_types(gpu, CudaMem, oracle)


@pytest.mark.gpu
def test_windows_indexes_gpu(gpu, oracle):
    run_indexes(gpu, CudaMem, oracle)


@pytest.mark.gpu
def test_windows_rejected_gpu(gpu, oracle):
    run_rejected(gpu, CudaMem, oracle)


@pytest.mark.gpu
def test_windows_damage_gpu(gpu, oracle):
    run_damage(gpu, CudaMem, oracle)


@pytest.mark.gpu
def test_windows_readahead_interleaved_gpu(gpu, oracle):
    run_readahead_interleaved(gpu, CudaMem, oracle)


@pytest.mark.gpu
def test_windows_decoder_paths_agree_gpu(gpu, oracle, monkeypatch):
    """the fused path, the split path and the throughput path give the same windows, and the throughput path runs"""
    pcm = harness.synth_pcm(n=BLOCK * 40 + 333, channels=2, bits=16, seed=81)
    data = oracle.encode(pcm, preset=6, block=BLOCK)
    full = gpu.decode(data)
    assert np.array_equal(full, pcm)
    idx = gpu.build_index(data)
    rng = np.random.default_rng(3)
    wins = [(int(s), int(ln)) for s, ln in zip(rng.integers(0, pcm.shape[1] - 5000, 40), rng.integers(0, 5000, 40))]
    wins += [(0, pcm.shape[1])]
    spec, room = layout(wins)
    outs = {}
    for path in ("fused", "split", "tput"):
        monkeypatch.setenv("LINNE_B200_SPLIT_DECODE", "1" if path == "split" else "0")
        dec = Decoder(gpu, 2)
        try:
            assert dec.index(padded(data), size=len(data))[0] == OK
            if path == "tput":
                dec.L.LINNEB200_DecoderSetThroughputBlocks(dec.h, 8)
            dec.L.LINNEB200_DecoderSetProfiling(dec.h, 1)
            rc, out, st = dec.windows(padded(data), len(data), idx, spec, 2, room)
            assert rc == OK and st == [OK] * len(spec)
            buf = (StageStat * 32)()
            m = dec.L.LINNEB200_DecoderGetStageStats(dec.h, buf, 32)
            names = {buf[i].name.decode() for i in range(m)}
            assert {"seek", "window_gather"} <= names, names
            if path == "tput":
                assert "tp_entropy" in names, names
            if path == "split":
                assert "stream_v2" not in names, names
            outs[path] = out
        finally:
            dec.close()
    assert np.array_equal(outs["fused"], expect(pcm, spec, 2, room))
    assert np.array_equal(outs["split"], outs["fused"]) and np.array_equal(outs["tput"], outs["fused"])


@pytest.mark.gpu
def test_windows_launch_count_does_not_grow_with_windows_gpu(gpu, oracle):
    pcm = harness.synth_pcm(n=BLOCK * 20, channels=2, bits=16, seed=91)
    data = oracle.encode(pcm, preset=3, block=BLOCK)
    idx = gpu.build_index(data)
    dec = Decoder(gpu, 2)
    try:
        assert dec.index(padded(data), size=len(data))[0] == OK
        counts = []
        rng = np.random.default_rng(4)
        for W in (1, 256):
            wins = [(int(s), 300) for s in rng.integers(0, pcm.shape[1] - 300, W)]
            wins[0] = (0, pcm.shape[1])                      # both sets need every block: the same batch
            spec, room = layout(wins, gap=0)
            before = dec.L.LINNEB200_DecoderLaunchCount(dec.h)
            rc, out, _ = dec.windows(padded(data), len(data), idx, spec, 2, room)
            counts.append(dec.L.LINNEB200_DecoderLaunchCount(dec.h) - before)
            assert rc == OK and np.array_equal(out, expect(pcm, spec, 2, room))
        assert counts[0] == counts[1], counts
    finally:
        dec.close()
