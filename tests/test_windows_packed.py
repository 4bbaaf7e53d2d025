"""LINNEB200_DecodeWindowsPacked: sample windows of a stream as the bytes of a WAV data chunk (interleaved little-endian
samples, as DecodeWholePacked writes them), and the command-line driver's excerpt options built on it.  Every window
must equal the same frames of DecodeWholePacked byte for byte, the bytes outside the windows (and of failed windows)
must keep their sentinel, and statuses and result codes must be those DecodeWindows gives for the same request.

CPU: the host code on the simulator.  GPU: the product."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import harness
from harness import OK, INVALID_ARGUMENT, INVALID_FORMAT, INSUFFICIENT_DATA, PARAMETER_NOT_SET, DATA_CORRUPTION
from linne_b200.api import StageStat, Window, index_points
from test_cli import B200_CLI, HOSTSIM_CLI, wav_data, write_wav
from test_windows import BLOCK, Decoder, layout, padded, shapes, stream_cases, u8


def sentinel(nbytes):
    """a byte pattern no decoder writes by accident"""
    return ((np.arange(nbytes, dtype=np.uint32) * 37 + 11) % 251).astype(np.uint8)


def frame_bytes(codec, data):
    hdr = codec.decode_header(data)[1]
    return hdr.num_channels * hdr.bits_per_sample // 8


def windows_packed(dec, data, size, index, spec, frame, room):
    """windows (first, len, out_offset) into `room` frames of packed PCM filled with the sentinel"""
    pts, npts = index_points(index)
    wins = (Window * max(1, len(spec)))(*[Window(s, n, o, 99) for s, n, o in spec])
    out = sentinel(max(1, room * frame))
    rc = dec.L.LINNEB200_DecodeWindowsPacked(dec.h, u8(data), size, pts, npts, wins, len(spec), u8(out), room)
    return rc, out, [wins[i].status for i in range(len(spec))]


def expect_packed(full, spec, frame, room, ok=None):
    want = sentinel(max(1, room * frame))
    for i, (s, n, o) in enumerate(spec):
        if ok is None or ok[i]:
            want[o * frame:(o + n) * frame] = np.frombuffer(full[s * frame:(s + n) * frame], np.uint8)
    return want


def check_exact(codec, data, spec_windows, full=None):
    full = codec.decode_packed(data) if full is None else full
    frame = frame_bytes(codec, data)
    spec, room = layout(spec_windows)
    room += 3                                                # bytes past the last window keep the sentinel too
    hdr = codec.decode_header(data)[1]
    dec = Decoder(codec, hdr.num_channels)
    try:
        host = padded(data)
        rc, idx, _ = dec.index(host, size=len(data))
        assert rc == OK
        rc, out, st = windows_packed(dec, host, len(data), idx, spec, frame, room)
        assert rc == OK and st == [OK] * len(spec), (rc, st)
        assert np.array_equal(out, expect_packed(full, spec, frame, room))
    finally:
        dec.close()


def run_streams(codec, oracle, channels, bits, preset, ms):
    pcm = harness.synth_pcm(n=BLOCK * 6 + 777, channels=channels, bits=bits, seed=40 + preset + channels)
    data = oracle.encode(pcm, bits=bits, preset=preset, block=BLOCK, ms=ms)
    full = codec.decode_packed(data)
    assert full == harness.pack_pcm(pcm, bits)
    check_exact(codec, data, shapes(pcm.shape[1], codec.build_index(data)), full)


def run_damage(codec, oracle):
    """the three damage cases of test_windows.run_damage: the statuses and result of DecodeWindows for the same request"""
    pcm = harness.synth_pcm(n=BLOCK * 6 + 300, channels=2, bits=16, seed=51)
    data = oracle.encode(pcm, preset=4, block=BLOCK)
    n = pcm.shape[1]
    full = harness.pack_pcm(pcm, 16)
    idx = codec.build_index(data)
    starts = [int(s) for s, _ in idx]
    windows = [(10, 50), (starts[2] + 5, 40), (starts[1] + 100, BLOCK), (starts[3] - 20, 40), (starts[4], 10), (0, n),
               (n - 5, 5), (7, 0)]
    spec, room = layout(windows)

    def run(image, size, index, check_crc=1):
        host = padded(bytes(image[:size]))
        dec = Decoder(codec, 2, check_crc)
        try:
            dec.L.LINNEDecoder_SetHeader(dec.h, C.byref(codec.decode_header(data)[1]))
            rc, out, st = windows_packed(dec, host, size, index, spec, 4, room)
            rc2, planes, st2 = dec.windows(host, size, index, spec, 2, room)
            assert rc == rc2 and st == st2, (rc, rc2, st, st2)
            # the OK windows hold DecodeWindows's samples (with CRC checks off, those of the damaged block too)
            want = sentinel(room * 4)
            for (s, ln, o), w in zip(spec, st):
                if w == OK:
                    want[o * 4:(o + ln) * 4] = np.frombuffer(harness.pack_pcm(planes[:, o:o + ln], 16), np.uint8)
            assert np.array_equal(out, want)
            if check_crc:
                assert np.array_equal(out, expect_packed(full, spec, 4, room, [w == OK for w in st]))
            return rc, st
        finally:
            dec.close()

    bad = bytearray(data)
    bad[int(idx[2][1]) + 40] ^= 0x10
    rc, st = run(bad, len(bad), idx)
    assert rc == DATA_CORRUPTION and OK in st, st
    assert run(bad, len(bad), idx, check_crc=0) == (OK, [OK] * len(spec))
    moved = idx.copy()
    moved[3][1] += 17
    rc, st = run(data, len(data), moved)
    assert rc == INVALID_FORMAT and OK in st, st
    rc, st = run(data, int(idx[-1][1]) + 20, idx)
    assert rc == INSUFFICIENT_DATA and OK in st, st


def run_rejected(codec, oracle):
    """test_windows.run_rejected's requests plus a capacity overflow: the result, an untouched buffer, no status"""
    pcm = harness.synth_pcm(n=BLOCK * 4 + 100, channels=2, bits=16, seed=31)
    data = oracle.encode(pcm, preset=1, block=BLOCK)
    n = pcm.shape[1]
    host = padded(data)
    fresh = Decoder(codec, 2)
    dec = Decoder(codec, 2)
    try:
        idx = codec.build_index(data)
        rc, out, st = windows_packed(fresh, host, len(data), idx, [(0, 10, 0)], 4, 16)
        assert rc == PARAMETER_NOT_SET and st == [99] and np.array_equal(out, sentinel(64))
        assert dec.index(host, size=len(data))[0] == OK

        def rejected(index, spec, room=64, want=INVALID_ARGUMENT):
            rc, out, st = windows_packed(dec, host, len(data), index, spec, 4, room)
            assert rc == want and st == [99] * len(spec) and np.array_equal(out, sentinel(room * 4)), (rc, st)
            assert dec.windows(host, len(data), index, spec, 2, room)[0] == want   # as DecodeWindows rejects it

        good = [(0, 10, 0), (n - 10, 10, 20)]
        rejected(idx, good + [(n - 5, 6, 40)])
        rejected(idx, good + [(0, 10, 60)])
        rejected(idx, good, room=29)                         # capacity overflow: 20 + 10 frames > 29
        bad = idx.copy(); bad[[1, 2]] = bad[[2, 1]]
        rejected(bad, good)
        bad = idx.copy(); bad[2][1] = bad[1][1]
        rejected(bad, good)
        bad = idx.copy(); bad[0][1] = 31
        rejected(bad, good)
        bad = idx.copy(); bad[0][0] = 1
        rejected(bad, good)
        bad = np.vstack([idx, [[n - 1, len(data)]]]).astype(np.uint32)
        rejected(bad, good)
        # exactly full is not an overflow, and the handle is still usable
        rc, out, st = windows_packed(dec, host, len(data), idx, good, 4, 30)
        assert rc == OK and np.array_equal(out, expect_packed(harness.pack_pcm(pcm, 16), good, 4, 30))
    finally:
        fresh.close()
        dec.close()


def run_python_api(codec, oracle):
    pcm = harness.synth_pcm(n=BLOCK * 3 + 10, channels=2, bits=24, seed=71)
    data = oracle.encode(pcm, bits=24, preset=0, block=BLOCK)
    full = harness.pack_pcm(pcm, 24)
    idx = codec.build_index(data)
    for index in (None, idx):
        got = codec.decode_windows_packed(data, [3, BLOCK - 1, 0], [10, 5, 0], index=index)
        assert got == [full[3 * 6:13 * 6], full[(BLOCK - 1) * 6:(BLOCK + 4) * 6], b""]
    rc, got, st = codec.decode_windows_packed(data, [0, len(pcm[0]) - 1], [5, 2], return_code=True)
    assert rc == INVALID_ARGUMENT and st == [0, 0]
    bad = bytearray(data)
    bad[int(idx[1][1]) + 40] ^= 0x10
    rc, got, st = codec.decode_windows_packed(bytes(bad), [0, BLOCK + 5], [5, 5], return_code=True)
    assert rc == DATA_CORRUPTION and st == [OK, DATA_CORRUPTION] and got[0] == full[:5 * 6]


def run_cli(cli, tmp_path):
    """-d --start S --length N: the WAV of the full decode, format for format, data bytes [S*F, (S+N)*F)"""
    cases = [(2, 16, 10240 * 2 + 2048, 11), (1, 24, 10240 + 4096, 12), (2, 8, 10240, 13)]
    pairs = []
    for ch, bits, n, seed in cases:
        pcm = harness.synth_pcm(n=n, channels=ch, bits=bits, seed=seed)
        wav = tmp_path / f"in_{seed}.wav"
        lnn = tmp_path / f"in_{seed}.lnn"
        write_wav(str(wav), pcm, bits)
        subprocess.run([cli, "-e", "-m", "2", str(wav), str(lnn)], check=True, capture_output=True, timeout=600)
        pairs.append((lnn, tmp_path / f"full_{seed}.wav", ch * bits // 8, n))
    subprocess.run([cli, "-d"] + [str(x) for p in pairs for x in p[:2]], check=True, capture_output=True, timeout=600)

    def check(opts, jobs, start, length):
        outs = [tmp_path / f"cut_{i}_{start}_{jobs}.wav" for i in range(len(pairs))]
        res = subprocess.run([cli, "-d", "-j", str(jobs)] + opts + [str(x) for p, o in zip(pairs, outs) for x in (p[0], o)],
                             capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr
        for (lnn, full, frame, n), out in zip(pairs, outs):
            fmt, body = wav_data(str(out))
            ffmt, fbody = wav_data(str(full))
            end = n if length is None else start + length
            assert fmt == ffmt and body == fbody[start * frame:end * frame]

    check(["--start", "9463", "--length", "777"], 1, 9463, 777)              # ends at the end of the shortest stream
    check(["--start", "10239"], 2, 10239, None)                 # to the end of every stream
    check(["--length", "5"], 2, 0, 5)
    check(["-c", "--start", "1", "--length", "10239"], 2, 1, 10239)
    # past the end of a stream: that file fails, with no output; the others are written
    short = tmp_path / "past.wav"
    ok = tmp_path / "ok.wav"
    res = subprocess.run([cli, "-d", "--start", "10240", "--length", "4096", str(pairs[2][0]), str(short), str(pairs[1][0]), str(ok)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode != 0 and "outside" in res.stderr and not short.exists()
    assert wav_data(str(ok))[1] == wav_data(str(pairs[1][1]))[1][10240 * 3:(10240 + 4096) * 3]
    # a damaged stream fails like a whole decode; -c decodes it
    bad = bytearray(pairs[0][0].read_bytes())
    bad[30 + 40] ^= 0x10
    bad_lnn = tmp_path / "bad.lnn"
    bad_lnn.write_bytes(bytes(bad))
    out = tmp_path / "bad.wav"
    res = subprocess.run([cli, "-d", "--start", "5", "--length", "100", str(bad_lnn), str(out)], capture_output=True, text=True, timeout=600)
    assert res.returncode != 0 and not out.exists()
    res = subprocess.run([cli, "-d", "-c", "--start", "5", "--length", "100", str(bad_lnn), str(out)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and out.exists()
    # usage errors
    for args in (["-e", "--start", "5", "a.wav", "b.lnn"], ["-e", "--length", "5", "a.wav", "b.lnn"],
                 ["-d", "--start", "x", "a.lnn", "b.wav"], ["-d", "--length"]):
        assert subprocess.run([cli] + args, capture_output=True, timeout=60).returncode != 0, args


# ---- the simulator -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("channels,bits,preset", stream_cases())
@pytest.mark.parametrize("ms", [0, 1])
def test_windows_packed_streams_hostsim(hostsim, oracle, channels, bits, preset, ms):
    if channels == 1 and ms:
        pytest.skip("M/S needs two channels")
    run_streams(hostsim, oracle, channels, bits, preset, ms)


def test_windows_packed_damage_hostsim(hostsim, oracle):
    run_damage(hostsim, oracle)


def test_windows_packed_rejected_hostsim(hostsim, oracle):
    run_rejected(hostsim, oracle)


def test_decode_windows_packed_python_api_hostsim(hostsim, oracle):
    run_python_api(hostsim, oracle)


@pytest.mark.skipif(not os.path.exists(HOSTSIM_CLI), reason="CLI binary not built")
def test_cli_excerpts_hostsim(tmp_path):
    run_cli(HOSTSIM_CLI, tmp_path)


# ---- the product ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("channels,bits,preset", stream_cases())
@pytest.mark.parametrize("ms", [0, 1])
def test_windows_packed_streams_gpu(gpu, oracle, channels, bits, preset, ms):
    if channels == 1 and ms:
        pytest.skip("M/S needs two channels")
    run_streams(gpu, oracle, channels, bits, preset, ms)


@pytest.mark.gpu
def test_windows_packed_damage_gpu(gpu, oracle):
    run_damage(gpu, oracle)


@pytest.mark.gpu
def test_windows_packed_rejected_gpu(gpu, oracle):
    run_rejected(gpu, oracle)


@pytest.mark.gpu
def test_decode_windows_packed_python_api_gpu(gpu, oracle):
    run_python_api(gpu, oracle)


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(B200_CLI), reason="CLI binary not built")
def test_cli_excerpts_gpu(tmp_path):
    run_cli(B200_CLI, tmp_path)


@pytest.mark.gpu
def test_windows_packed_decoder_paths_agree_gpu(gpu, oracle, monkeypatch):
    """fused, split and throughput paths give the same bytes; the call runs seek and the packed gather, no other
    conversion or gather"""
    pcm = harness.synth_pcm(n=BLOCK * 40 + 333, channels=2, bits=16, seed=81)
    data = oracle.encode(pcm, preset=6, block=BLOCK)
    full = harness.pack_pcm(pcm, 16)
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
            dec.L.LINNEB200_DecoderResetStageStats(dec.h)
            rc, out, st = windows_packed(dec, padded(data), len(data), idx, spec, 4, room)
            assert rc == OK and st == [OK] * len(spec)
            buf = (StageStat * 32)()
            m = dec.L.LINNEB200_DecoderGetStageStats(dec.h, buf, 32)
            names = {buf[i].name.decode() for i in range(m)}
            assert {"seek", "window_gather_packed"} <= names, names
            assert not {"pack_pcm", "window_gather"} & names, names
            if path == "tput":
                assert "tp_entropy" in names, names
            outs[path] = out
        finally:
            dec.close()
    assert np.array_equal(outs["fused"], expect_packed(full, spec, 4, room))
    assert np.array_equal(outs["split"], outs["fused"]) and np.array_equal(outs["tput"], outs["fused"])


@pytest.mark.gpu
def test_windows_packed_launch_count_gpu(gpu, oracle):
    """as many launches as DecodeWindows for the same windows, and as many for 1 window as for 256"""
    pcm = harness.synth_pcm(n=BLOCK * 20, channels=2, bits=16, seed=91)
    data = oracle.encode(pcm, preset=3, block=BLOCK)
    full = harness.pack_pcm(pcm, 16)
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
            rc, out, _ = windows_packed(dec, padded(data), len(data), idx, spec, 4, room)
            packed = dec.L.LINNEB200_DecoderLaunchCount(dec.h) - before
            assert rc == OK and np.array_equal(out, expect_packed(full, spec, 4, room))
            before = dec.L.LINNEB200_DecoderLaunchCount(dec.h)
            assert dec.windows(padded(data), len(data), idx, spec, 2, room)[0] == OK
            assert packed == dec.L.LINNEB200_DecoderLaunchCount(dec.h) - before
            counts.append(packed)
        assert counts[0] == counts[1], counts
    finally:
        dec.close()
