"""Salvage decodes: every intact block of a damaged stream, placed where it belongs, and a report of what was lost.

LINNEB200_DecodeSalvage / DecodeSalvagePacked (include/linne_b200.h) run a resynchronising scan over the image, verify
the candidates' CRCs, walk the verified blocks and decode the ones they can place.  Checked here, on the simulator and on
the GPU:
  - intact streams (every golden stream and the framing test's source stream) give OK, no records, and exactly what
    DecodeWhole / DecodeWholePacked give;
  - a matrix of damage on the 7-block source stream of test_decode_framing (B = 1024: compressed blocks, a silent block 1,
    a raw block 3, a 300-sample tail 6) gives literal records; samples outside the records equal the intact decode,
    samples inside are zero, and the packed bytes are the packed form of those planes;
  - segments that cannot be anchored are not decoded: a middle segment between gaps that cost 0 and 2 blocks, a last
    segment that does not end with the tail block, a last segment that would overlap the first;
  - a well-formed block with a correct CRC planted inside damage, with nothing verified behind it, is not accepted;
  - lost frames of 8-bit packed output are the biased silence 128;
  - rejected requests write nothing;
  - the command-line driver's -F and the Python wrappers agree with the C calls;
  - a stream of 3000 blocks with 64 payload flips and two framing gaps (on the GPU through the throughput kernels)."""
import ctypes as C
import subprocess

import numpy as np
import pytest

import harness
from harness import OK, INVALID_ARGUMENT, INSUFFICIENT_BUFFER, PARAMETER_NOT_SET, LINNEDecoderConfig
from linne_b200.api import Damage, StageStat
from test_cli import wav_data, HOSTSIM_CLI, B200_CLI
from test_decode_framing import source, block_offsets, fix_crc, BLOCK, FRAMES

INVALID_FORMAT, INSUFFICIENT_DATA, CORRUPT = 2, 4, 6
u8p = C.POINTER(C.c_uint8)
B = BLOCK


def u8(a):
    return a.ctypes.data_as(u8p)


GARBAGE = bytes((i * 7 + 3) % 251 for i in range(37))      # no 0xFF: no sync code in it


def damaged(oracle, good, case):
    """the image of one row of the matrix"""
    offs = block_offsets(good)
    b = bytearray(good)
    if case == "payload_2":
        b[offs[2] + 40] ^= 0x10
    elif case == "payload_0_and_tail":
        b[offs[0] + 40] ^= 0x10
        b[offs[6] + 40] ^= 0x10
    elif case == "sync_2":
        b[offs[2]] ^= 0x01
    elif case == "size_2_into_4":
        b[offs[2] + 2:offs[2] + 6] = (offs[4] + 100 - offs[2] - 6).to_bytes(4, "big")
    elif case == "delete_100_in_3":
        del b[offs[3] + 200:offs[3] + 300]
    elif case == "insert_37_between_3_4":
        b[offs[4]:offs[4]] = GARBAGE
    elif case == "truncate_in_4":
        del b[offs[4] + 500:]
    elif case == "truncate_before_6":
        del b[offs[6]:]
    elif case == "sync_1_and_4":
        b[offs[1]] ^= 0x01
        b[offs[4]] ^= 0x01
    elif case == "sync_1_and_cut_3_to_4":
        b[offs[1]] ^= 0x01
        del b[offs[3] + 300:offs[4] + 300]
    elif case == "sync_tail":
        b[offs[6] + 1] ^= 0x80
    elif case == "planted_block_in_2":
        # sync of block 2 damaged; inside its payload a silent block of B samples with a correct CRC whose successor
        # (11 bytes on) is payload: verified, never confirmed
        b[offs[2]] ^= 0x01
        p = offs[2] + 20
        b[p:p + 11] = b"\xff\xff" + (5).to_bytes(4, "big") + b"\0\0" + bytes([1]) + B.to_bytes(2, "big")
        fix_crc(oracle, b, p)
    elif case == "insert_37_before_2_and_sync_4":
        # gaps that cost 0 and 2 blocks: the middle segment (blocks 2, 3) cannot be placed
        b[offs[4]] ^= 0x01
        b[offs[2]:offs[2]] = GARBAGE
    elif case == "sync_2_and_truncate_before_5":
        # the chain behind the gap ends at the image's end, but with a full block, not the 300-sample tail: no back anchor
        b[offs[2]] ^= 0x01
        del b[offs[5]:]
    elif case == "repeat_2_after_garbage":
        # blocks 0-3, garbage, blocks 2-6 again: the last segment would overlap the first, so it is not placed
        b[offs[4]:] = GARBAGE + bytes(good[offs[2]:])
    elif case == "zeroed_header":
        b[:30] = bytes(30)
    else:
        assert case == "intact"
    return bytes(b)


# (first_sample, num_samples, byte_offset, byte_size, status) per record; intact offsets:
# 30, 2747, 2758 (block 1 is 11 silent bytes), 5378, 9485 (block 3 is raw), 11999, 14548, end 15420
EXPECTED = {
    "intact": (OK, []),
    "zeroed_header": (OK, []),
    "payload_2": (CORRUPT, [(2048, 1024, 2758, 2620, CORRUPT)]),
    "payload_0_and_tail": (CORRUPT, [(0, 1024, 30, 2717, CORRUPT), (6144, 300, 14548, 872, CORRUPT)]),
    "sync_2": (CORRUPT, [(2048, 1024, 2758, 2620, INVALID_FORMAT)]),
    "size_2_into_4": (CORRUPT, [(2048, 1024, 2758, 2620, CORRUPT)]),
    "delete_100_in_3": (CORRUPT, [(3072, 1024, 5378, 4007, CORRUPT)]),
    "insert_37_between_3_4": (CORRUPT, [(4096, 0, 9485, 37, INVALID_FORMAT)]),
    "truncate_in_4": (CORRUPT, [(4096, 2348, 9485, 500, INSUFFICIENT_DATA)]),
    "truncate_before_6": (CORRUPT, [(6144, 300, 14548, 0, INSUFFICIENT_DATA)]),
    "sync_1_and_4": (CORRUPT, [(1024, 1024, 2747, 11, INVALID_FORMAT), (4096, 1024, 9485, 2514, INVALID_FORMAT)]),
    "sync_1_and_cut_3_to_4": (CORRUPT, [(1024, 4096, 2747, 5145, INVALID_FORMAT)]),
    "sync_tail": (CORRUPT, [(6144, 300, 14548, 872, INVALID_FORMAT)]),
    "planted_block_in_2": (CORRUPT, [(2048, 1024, 2758, 2620, INVALID_FORMAT)]),
    "insert_37_before_2_and_sync_4": (CORRUPT, [(2048, 3072, 2758, 9278, INVALID_FORMAT)]),
    "sync_2_and_truncate_before_5": (CORRUPT, [(2048, 4396, 2758, 9241, INVALID_FORMAT)]),
    "repeat_2_after_garbage": (CORRUPT, [(4096, 2348, 9485, 12699, INVALID_FORMAT)]),
}
CASES = list(EXPECTED)


class Handle:
    """a decoder handle with a header latched (the stream's own unless one is given)"""

    def __init__(self, codec, header, channels=2, check_crc=1):
        self.L = codec.lib
        self.h = self.L.LINNEDecoder_Create(C.byref(LINNEDecoderConfig(channels, 3, 128, check_crc)), None, 0)
        assert self.h
        if header is not None:
            assert self.L.LINNEDecoder_SetHeader(self.h, C.byref(header)) == OK

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.L.LINNEDecoder_Destroy(self.h)


def salvage_c(codec, img, header, cap=64):
    """both C calls on one handle -> (rc, planes, records), (rc, packed bytes, records)"""
    C_, N, bits = header.num_channels, header.num_samples, header.bits_per_sample
    nbytes = N * C_ * (bits // 8)
    buf = np.frombuffer(img, np.uint8)
    with Handle(codec, header, max(C_, 2)) as d:
        out = np.full((C_, N + 8), 0x5A5A5A5A, np.int32)
        dmg, n = (Damage * cap)(), C.c_uint32(99)
        rc = d.L.LINNEB200_DecodeSalvage(d.h, u8(buf), len(img), harness._chan_ptrs(out), C_, N, dmg, cap, C.byref(n))
        assert np.all(out[:, N:] == 0x5A5A5A5A)                     # nothing past N samples
        planes = (rc, out[:, :N].copy(), [tuple(getattr(r, f) for f, _ in Damage._fields_) for r in dmg[:n.value]])
        raw = np.full(nbytes + 64, 0xA5, np.uint8)
        dmg, n = (Damage * cap)(), C.c_uint32(99)
        rc = d.L.LINNEB200_DecodeSalvagePacked(d.h, u8(buf), len(img), u8(raw), N, dmg, cap, C.byref(n))
        assert np.all(raw[nbytes:] == 0xA5)
        packed = (rc, raw[:nbytes].tobytes(), [tuple(getattr(r, f) for f, _ in Damage._fields_) for r in dmg[:n.value]])
    return planes, packed


def lost_mask(records, n):
    m = np.zeros(n, bool)
    for s, k, _, _, _ in records:
        m[s:s + k] = True
    return m


def check_output(planes, packed, want_pcm, bits, records):
    lost = lost_mask(records, want_pcm.shape[1])
    assert np.array_equal(planes[:, ~lost], want_pcm[:, ~lost])
    assert np.all(planes[:, lost] == 0)
    assert packed == harness.pack_pcm(planes, bits)


def check_case(codec, oracle, case):
    pcm, good = source(oracle)
    img = damaged(oracle, good, case)
    header = codec.decode_header(good)[1]                           # the intact stream's parameters, latched
    want_rc, want_rec = EXPECTED[case]
    (rc, planes, rec), (prc, packed, prec) = salvage_c(codec, img, header)
    assert (rc, rec) == (want_rc, want_rec)
    assert (prc, prec) == (want_rc, want_rec)
    check_output(planes, packed, pcm, 16, rec)
    # the Python wrappers: the image's own header, or the given one where the image's is gone
    given = header if case == "zeroed_header" else None
    assert codec.decode_salvage(img, given)[0::2] == (want_rc, want_rec)
    assert np.array_equal(codec.decode_salvage(img, given)[1], planes)
    assert codec.decode_salvage_packed(img, given) == (want_rc, packed, want_rec)


def check_intact(codec, oracle):
    """every golden stream and the framing source: OK, no records, DecodeWhole's planes and DecodeWholePacked's bytes"""
    streams = [bytes(harness.load_golden(g)["stream"]) for g in harness.GOLDEN_CASES + ["mixed_types_m5"]]
    streams.append(source(oracle)[1])
    for data in streams:
        rc, header = codec.decode_header(data)
        assert rc == OK
        (rc, planes, rec), (prc, packed, prec) = salvage_c(codec, data, header)
        assert (rc, rec, prc, prec) == (OK, [], OK, [])
        assert np.array_equal(planes, codec.decode(data))
        assert packed == codec.decode_packed(data)


def check_8bit_packed(codec, oracle):
    """8-bit packed output: lost frames are the biased silence 128"""
    pcm = harness.synth_pcm(n=4 * B + 100, channels=1, bits=8, seed=41)
    good = oracle.encode(pcm, bits=8, preset=3, block=B)
    offs = block_offsets(good) + [len(good)]
    assert good[offs[1] + 8] == 0 and offs[2] - offs[1] > 64              # block 1 is compressed
    b = bytearray(good)
    b[offs[1] + 40] ^= 0x04
    header = codec.decode_header(good)[1]
    (rc, planes, rec), (prc, packed, prec) = salvage_c(codec, bytes(b), header)
    want = [(1024, 1024, offs[1], offs[2] - offs[1], CORRUPT)]
    assert (rc, rec, prc, prec) == (CORRUPT, want, CORRUPT, want)
    check_output(planes, packed, pcm, 8, rec)
    raw = np.frombuffer(packed, np.uint8)
    assert np.all(raw[1024:2048] == 128) and np.array_equal(raw[:1024], np.frombuffer(harness.pack_pcm(pcm, 8), np.uint8)[:1024])


def check_rejections(codec, oracle):
    pcm, good = source(oracle)
    header = codec.decode_header(good)[1]
    buf = np.frombuffer(good, np.uint8)
    out = np.full((2, FRAMES), 7, np.int32)
    raw = np.full(FRAMES * 4, 7, np.uint8)
    dmg, n = (Damage * 4)(), C.c_uint32(99)
    L = codec.lib
    with Handle(codec, None) as d:                                  # no header latched
        assert L.LINNEB200_DecodeSalvage(d.h, u8(buf), len(good), harness._chan_ptrs(out), 2, FRAMES, dmg, 4, C.byref(n)) == PARAMETER_NOT_SET
        assert L.LINNEB200_DecodeSalvagePacked(d.h, u8(buf), len(good), u8(raw), FRAMES, dmg, 4, C.byref(n)) == PARAMETER_NOT_SET
    with Handle(codec, header) as d:
        assert L.LINNEB200_DecodeSalvage(d.h, None, len(good), harness._chan_ptrs(out), 2, FRAMES, dmg, 4, C.byref(n)) == INVALID_ARGUMENT
        assert L.LINNEB200_DecodeSalvage(d.h, u8(buf), len(good), harness._chan_ptrs(out), 2, FRAMES, None, 4, C.byref(n)) == INVALID_ARGUMENT
        assert L.LINNEB200_DecodeSalvage(d.h, u8(buf), len(good), harness._chan_ptrs(out), 2, FRAMES, dmg, 4, None) == INVALID_ARGUMENT
        assert L.LINNEB200_DecodeSalvagePacked(d.h, u8(buf), len(good), None, FRAMES, dmg, 4, C.byref(n)) == INVALID_ARGUMENT
        assert L.LINNEB200_DecodeSalvage(d.h, u8(buf), len(good), harness._chan_ptrs(out), 1, FRAMES, dmg, 4, C.byref(n)) == INSUFFICIENT_BUFFER
        assert L.LINNEB200_DecodeSalvage(d.h, u8(buf), len(good), harness._chan_ptrs(out), 2, FRAMES - 1, dmg, 4, C.byref(n)) == INSUFFICIENT_BUFFER
        assert L.LINNEB200_DecodeSalvagePacked(d.h, u8(buf), len(good), u8(raw), FRAMES - 1, dmg, 4, C.byref(n)) == INSUFFICIENT_BUFFER
        assert np.all(out == 7) and np.all(raw == 7) and n.value == 99
        # no room for records: the count still comes back, the output is complete
        img = damaged(oracle, good, "sync_1_and_4")
        ibuf = np.frombuffer(img, np.uint8)
        assert L.LINNEB200_DecodeSalvage(d.h, u8(ibuf), len(img), harness._chan_ptrs(out), 2, FRAMES, None, 0, C.byref(n)) == CORRUPT
        assert n.value == 2
        assert L.LINNEB200_DecodeSalvage(d.h, u8(ibuf), len(img), harness._chan_ptrs(out), 2, FRAMES, dmg, 1, C.byref(n)) == CORRUPT
        assert n.value == 2 and (dmg[0].first_sample, dmg[1].first_sample) == (1024, 0)
    check_output(out, harness.pack_pcm(out, 16), pcm, 16, EXPECTED["sync_1_and_4"][1])


def check_cli(cli, codec, oracle, tmp_path):
    pcm, good = source(oracle)
    img = damaged(oracle, good, "sync_1_and_4")
    (tmp_path / "bad.lnn").write_bytes(img)
    (tmp_path / "good.lnn").write_bytes(good)
    bad, ok, out_bad, out_ok = (str(tmp_path / f) for f in ("bad.lnn", "good.lnn", "bad.wav", "good.wav"))
    header = codec.decode_header(good)[1]
    _, packed = salvage_c(codec, img, header)
    res = subprocess.run([cli, "-d", "-F", bad, out_bad, ok, out_ok, "-j", "1"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 2, res.stderr
    assert wav_data(out_bad)[1] == packed[1] and len(packed[1]) == FRAMES * 4
    assert wav_data(out_ok)[1] == harness.pack_pcm(pcm, 16)
    lines = [l for l in res.stderr.splitlines() if "lost" in l]
    assert lines == [f"{bad}: frames [1024, 2048) lost, bytes [2747, 2758): INVALID_FORMAT",
                     f"{bad}: frames [4096, 5120) lost, bytes [9485, 11999): INVALID_FORMAT"]
    # intact files only: exit code 0
    res = subprocess.run([cli, "-d", "-F", ok, out_ok], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "lost" not in res.stderr
    # without -F nothing changes: the damaged file fails
    res = subprocess.run([cli, "-d", bad, out_bad], capture_output=True, text=True, timeout=600)
    assert res.returncode == 1 and "decode failed (2)" in res.stderr
    # -F does not combine with an excerpt
    res = subprocess.run([cli, "-d", "-F", "--start", "10", ok, out_ok], capture_output=True, text=True, timeout=600)
    assert res.returncode == 1 and "-F" in res.stderr


# ---- the simulator -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_salvage_matrix_hostsim(hostsim, oracle, case):
    check_case(hostsim, oracle, case)


def test_salvage_intact_hostsim(hostsim, oracle):
    check_intact(hostsim, oracle)


def test_salvage_rejections_hostsim(hostsim, oracle):
    check_rejections(hostsim, oracle)


def test_salvage_8bit_packed_hostsim(hostsim, oracle):
    check_8bit_packed(hostsim, oracle)


def test_salvage_cli_hostsim(hostsim, oracle, tmp_path):
    check_cli(HOSTSIM_CLI, hostsim, oracle, tmp_path)


# ---- the product ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_salvage_matrix_gpu(gpu, oracle, case):
    check_case(gpu, oracle, case)


@pytest.mark.gpu
def test_salvage_intact_gpu(gpu, oracle):
    check_intact(gpu, oracle)


@pytest.mark.gpu
def test_salvage_rejections_gpu(gpu, oracle):
    check_rejections(gpu, oracle)


@pytest.mark.gpu
def test_salvage_8bit_packed_gpu(gpu, oracle):
    check_8bit_packed(gpu, oracle)


@pytest.mark.gpu
def test_salvage_cli_gpu(gpu, oracle, tmp_path):
    check_cli(B200_CLI, gpu, oracle, tmp_path)


def check_scale(codec, oracle, want_stages):
    """3000 blocks of 1024 samples, 64 seeded payload flips and two sync flips (the flips keep two blocks away from the
    sync flips: a framing gap is only recovered from when the block behind it is confirmed): the records and samples
    follow from the intact decode block by block"""
    clip = harness.synth_pcm(n=30 * B, channels=2, bits=16, seed=23)
    good = harness.tile_stream(oracle.encode(clip, preset=3, block=B), 100, B)
    offs = block_offsets(good) + [len(good)]
    nb = len(offs) - 1
    assert nb == 3000
    header = codec.decode_header(good)[1]
    intact = codec.decode(good)
    rng = np.random.default_rng(31)
    gaps = [1000, 2000]
    allowed = [k for k in range(nb - 2) if all(abs(k - g) > 2 for g in gaps) and offs[k + 1] - offs[k] > 64]
    flips = sorted(rng.choice(allowed, size=64, replace=False).tolist())
    b = bytearray(good)
    for k in flips:
        b[offs[k] + 11 + int(rng.integers(0, offs[k + 1] - offs[k] - 11))] ^= 1 << int(rng.integers(0, 8))
    for k in gaps:
        b[offs[k]] ^= 0x01
    status = {k: CORRUPT for k in flips} | {k: INVALID_FORMAT for k in gaps}
    want = []
    for k in sorted(status):                                        # runs of damaged blocks merge into one record
        if want and want[-1][0] + want[-1][1] == k * B:
            s, n, o, size, st = want[-1]
            want[-1] = (s, n + B, o, size + offs[k + 1] - offs[k], st)
        else:
            want.append((k * B, B, offs[k], offs[k + 1] - offs[k], status[k]))
    img = np.frombuffer(bytes(b), np.uint8)
    with Handle(codec, header) as d:
        d.L.LINNEB200_DecoderSetThroughputBlocks(d.h, 64)
        d.L.LINNEB200_DecoderSetProfiling(d.h, 1)
        out = np.zeros((2, header.num_samples), np.int32)
        dmg, n = (Damage * 256)(), C.c_uint32(0)
        rc = d.L.LINNEB200_DecodeSalvage(d.h, u8(img), len(img), harness._chan_ptrs(out), 2, header.num_samples, dmg, 256, C.byref(n))
        buf = (StageStat * 32)()
        stages = {buf[i].name.decode() for i in range(d.L.LINNEB200_DecoderGetStageStats(d.h, buf, 32))}
    assert want_stages <= stages, stages
    rec = [tuple(getattr(r, f) for f, _ in Damage._fields_) for r in dmg[:n.value]]
    assert (rc, rec) == (CORRUPT, want)
    check_output(out, harness.pack_pcm(out, 16), intact, 16, rec)


def test_salvage_scale_hostsim(hostsim, oracle):
    check_scale(hostsim, oracle, set())


@pytest.mark.gpu
def test_salvage_scale_throughput_gpu(gpu, oracle):
    """the same through the throughput kernels"""
    check_scale(gpu, oracle, {"tp_entropy", "tp_synth", "resync_scan", "salvage_crc"})
