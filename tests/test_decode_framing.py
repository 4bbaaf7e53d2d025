"""Stream framing through every decode entry point.

Every entry point that reads a stream hops over its block headers (sync code, size, type, sample count) before the
kernels run, and must stop at the same block with the same result as the reference's per-block checks
(linne_decoder.c:604-653, :383).  A matrix of damaged oracle streams goes through DecodeWhole, DecodeWholePacked, the
DecodeBlock loop (with and without read-ahead), DecodeWholeResident (with a host copy and with the image in device memory
only), DecodeFilesResident, DecodeFilesPacked and BuildIndex (host and device image).  The expected values are literal:
result code, frames that equal the undamaged decode, and frames written at all (the rest of the buffer keeps its
sentinel).  Where entry points differ, the table records the difference.

Streams of many tiny silent blocks (11 bytes each) must decode through the corpus and device-image entry points too.

CPU: the host code on the simulator (its "device" memory is host memory).  GPU: the product, buffers in HBM."""
import ctypes as C

import numpy as np
import pytest

import harness
from harness import OK, LINNEDecoderConfig
from linne_b200.api import FileDesc, SeekPoint
from test_corpus_batches import HostMem, CudaMem

BLOCK = 1024
FRAMES = BLOCK * 6 + 300
SENTINEL = 0x5A5A5A5A                 # outside every sample range
PACKED_SENTINEL = 0xA5
u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)


def u8(a):
    return a.ctypes.data_as(u8p)


def padded(data, size=None):
    size = len(data) if size is None else size
    buf = np.zeros(size + 16, np.uint8)
    buf[:size] = np.frombuffer(bytes(data[:size]), np.uint8)
    return buf


def source(oracle):
    """stereo 16-bit: compressed blocks 0, 2, 4, 5, a silent block 1, a raw block (full-scale noise) 3, a tail block 6"""
    rng = np.random.default_rng(5)
    pcm = harness.synth_pcm(n=FRAMES, channels=2, bits=16, seed=17)
    pcm[:, BLOCK:2 * BLOCK] = 0
    pcm[:, 3 * BLOCK:4 * BLOCK] = rng.integers(-32768, 32768, size=(2, BLOCK), dtype=np.int32)
    return pcm, oracle.encode(pcm, preset=3, block=BLOCK)


def block_offsets(data):
    off, out = 30, []
    while off < len(data):
        out.append(off)
        off += 6 + int.from_bytes(data[off + 2:off + 6], "big")
    return out


def fix_crc(oracle, data, off):
    end = off + 6 + int.from_bytes(data[off + 2:off + 6], "big")
    data[off + 6:off + 8] = oracle.crc16(bytes(data[off + 8:end])).to_bytes(2, "big")


def damaged(oracle, data, case):
    """(image, size, check_crc) of one row of the matrix"""
    offs = block_offsets(data)
    b = bytearray(data)
    size, crc = len(data), 1
    if case == "bad_sync":
        b[offs[2]] ^= 0x01
    elif case == "cut_in_size":
        size = offs[2] + 4
    elif case == "cut_in_payload":
        size = offs[2] + 40
    elif case == "size_below_5":
        b[offs[2] + 2:offs[2] + 6] = (4).to_bytes(4, "big")
    elif case in ("type9_crc_on", "type9_crc_off"):
        b[offs[2] + 8] = 9
        crc = 1 if case == "type9_crc_on" else 0
    elif case == "raw_cut":
        assert b[offs[3] + 8] == 2
        size = offs[3] + 11 + 100
    elif case == "too_many_samples":
        b[offs[2] + 9:offs[2] + 11] = (0xFFFF).to_bytes(2, "big")
        fix_crc(oracle, b, offs[2])
    elif case == "crc_mismatch":
        b[offs[2] + 40] ^= 0x10
    elif case == "ends_on_boundary":
        size = offs[4]
    else:
        assert case == "intact"
    return bytes(b[:size]), size, crc


def prefix_and_written(out, want):
    """frames (columns) equal to the undamaged decode from the start, and one past the last frame that was written"""
    n = min(out.shape[1], want.shape[1])
    same = np.all(out[:, :n] == want[:, :n], axis=0)
    k = int(np.argmin(same)) if not same.all() else n
    touched = np.nonzero(np.any(out != SENTINEL, axis=0))[0]
    return k, int(touched[-1]) + 1 if len(touched) else 0


def packed_planes(raw, frames, channels):
    """int16 interleaved bytes -> int32 planes; a frame whose bytes all kept the sentinel reads as SENTINEL"""
    b = raw[:frames * channels * 2].reshape(frames, channels * 2)
    pcm = b.view("<i2").astype(np.int32).T.copy()
    pcm[:, np.all(b == PACKED_SENTINEL, axis=1)] = SENTINEL
    return pcm


class Decoder:
    def __init__(self, codec, check_crc, readahead=0):
        self.L = codec.lib
        self.h = self.L.LINNEDecoder_Create(C.byref(LINNEDecoderConfig(2, 3, 128, check_crc)), None, 0)
        assert self.h
        if readahead:
            self.L.LINNEB200_DecoderSetReadahead(self.h, readahead)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.L.LINNEDecoder_Destroy(self.h)


def run_whole(codec, Mem, img, size, crc, want):
    out = np.full((2, FRAMES), SENTINEL, np.int32)
    with Decoder(codec, crc) as d:
        rc = d.L.LINNEDecoder_DecodeWhole(d.h, u8(img), size, harness._chan_ptrs(out), 2, FRAMES)
    return (rc, *prefix_and_written(out, want))


def run_whole_packed(codec, Mem, img, size, crc, want):
    raw = np.full(FRAMES * 4 + 64, PACKED_SENTINEL, np.uint8)
    frames = C.c_uint32(12345)
    with Decoder(codec, crc) as d:
        rc = d.L.LINNEB200_DecodeWholePacked(d.h, u8(img), size, u8(raw), FRAMES, C.byref(frames))
    assert np.all(raw[FRAMES * 4:] == PACKED_SENTINEL)
    return (rc, frames.value, *prefix_and_written(packed_planes(raw, FRAMES, 2), want))


def block_loop(codec, img, size, crc, want, readahead):
    """a player: one DecodeBlock per call with room for one block, from after the header until the stream ends"""
    out = np.full((2, FRAMES + 2 * BLOCK), SENTINEL, np.int32)
    rc, off, done = OK, 30, 0
    with Decoder(codec, crc, readahead) as d:
        assert d.L.LINNEDecoder_SetHeader(d.h, C.byref(codec.decode_header(img[:30].tobytes())[1])) == OK
        for _ in range(64):
            if done >= FRAMES or off >= size:
                break
            ptrs = (i32p * 2)(*[out[c, done:].ctypes.data_as(i32p) for c in range(2)])
            used, got = C.c_uint32(0), C.c_uint32(0)
            rc = d.L.LINNEDecoder_DecodeBlock(d.h, u8(img[off:]), size - off, ptrs, 2, BLOCK, C.byref(used), C.byref(got))
            done += got.value
            if rc != OK:
                break
            off += used.value
    return (rc, done, *prefix_and_written(out, want))


def run_block_loop(codec, Mem, img, size, crc, want):
    return block_loop(codec, img, size, crc, want, 0)


def run_block_loop_readahead(codec, Mem, img, size, crc, want):
    return block_loop(codec, img, size, crc, want, 4)


def resident(codec, Mem, img, size, crc, want, host_copy):
    stride = FRAMES + 4
    d_pcm = Mem(np.full((2, stride), SENTINEL, np.int32))
    d_img = Mem(img)
    with Decoder(codec, crc) as d:
        rc = d.L.LINNEB200_DecodeWholeResident(d.h, u8(img) if host_copy else None, C.c_void_p(d_img.ptr), size,
                                               C.c_void_p(d_pcm.ptr), stride, 2, FRAMES)
    return (rc, *prefix_and_written(d_pcm.get(), want))


def run_resident_host(codec, Mem, img, size, crc, want):
    return resident(codec, Mem, img, size, crc, want, True)


def run_resident_device(codec, Mem, img, size, crc, want):
    return resident(codec, Mem, img, size, crc, want, False)


def corpus(img, size, good):
    """the damaged stream, then the intact one 16-aligned behind it"""
    second = (size + 15) // 16 * 16
    image = np.zeros(second + len(good) + 16, np.uint8)
    image[:size] = img[:size]
    image[second:second + len(good)] = np.frombuffer(good, np.uint8)
    return image, second


def run_files_resident(codec, Mem, img, size, crc, want, good):
    image, second = corpus(img, size, good)
    stride = 2 * FRAMES + 8
    files = (FileDesc * 2)(FileDesc(0, FRAMES, 0, size, 99), FileDesc(FRAMES + 4, FRAMES, second, len(good), 99))
    d_pcm = Mem(np.full((2, stride), SENTINEL, np.int32))
    d_img = Mem(image)
    with Decoder(codec, crc) as d:
        rc = d.L.LINNEB200_DecodeFilesResident(d.h, C.c_void_p(d_img.ptr), second + len(good), files, 2,
                                               C.c_void_p(d_pcm.ptr), stride)
    out = d_pcm.get()
    if files[1].status == OK:
        assert np.array_equal(out[:, FRAMES + 4:2 * FRAMES + 4], want)
    return (rc, files[0].status, files[1].status, *prefix_and_written(out[:, :FRAMES + 4], want))


def run_files_packed(codec, Mem, img, size, crc, want, good):
    """a failed file's frames are undefined here: only the statuses and the intact file's frames are checked"""
    image, second = corpus(img, size, good)
    files = (FileDesc * 2)(FileDesc(0, FRAMES, 0, size, 99), FileDesc(0, FRAMES, second, len(good), 99))
    raw = np.full(2 * FRAMES * 4 + 64, PACKED_SENTINEL, np.uint8)
    with Decoder(codec, crc) as d:
        rc = d.L.LINNEB200_DecodeFilesPacked(d.h, u8(image), second + len(good), files, 2, u8(raw))
    if files[1].status == OK:
        assert files[1].first_sample == FRAMES
        assert np.array_equal(packed_planes(raw[FRAMES * 4:], FRAMES, 2), want)
    return (rc, files[0].status, files[1].status)


def index(codec, Mem, img, size, crc, want, good_index, on_device):
    pts = (SeekPoint * 16)()
    n = C.c_uint32(0)
    with Decoder(codec, crc) as d:
        if on_device:
            d_img = Mem(img)
            rc = d.L.LINNEB200_DecoderBuildIndex(d.h, None, C.c_void_p(d_img.ptr), size, pts, 16, C.byref(n))
        else:
            rc = d.L.LINNEB200_DecoderBuildIndex(d.h, u8(img), None, size, pts, 16, C.byref(n))
    got = np.frombuffer(bytes(pts), np.uint32).reshape(-1, 2)[:n.value]
    assert np.array_equal(got, good_index[:n.value])
    return (rc, n.value)


ENTRY_POINTS = ["whole", "whole_packed", "block_loop", "block_loop_readahead", "resident_host", "resident_device",
                "files_resident", "files_packed", "index_host", "index_device"]

# result codes: 0 OK, 2 INVALID_FORMAT, 3 INSUFFICIENT_BUFFER, 4 INSUFFICIENT_DATA, 6 DETECT_DATA_CORRUPTION
# whole, resident_*:   (rc, frames equal to the intact decode, frames written)
# whole_packed, block_loop*: (rc, frames reported, frames equal, frames written)
# files_resident:      (rc, status of the damaged file, status of the intact one, frames equal, frames written)
# files_packed:        (rc, status of the damaged file, status of the intact one)
# index_*:             (rc, seek points)
EXPECTED = {
    "intact": {"whole": (0, 6444, 6444), "whole_packed": (0, 6444, 6444, 6444), "block_loop": (0, 6444, 6444, 6444),
        "block_loop_readahead": (0, 6444, 6444, 6444), "resident_host": (0, 6444, 6444),
        "resident_device": (0, 6444, 6444), "files_resident": (0, 0, 0, 6444, 6444), "files_packed": (0, 0, 0),
        "index_host": (0, 7), "index_device": (0, 7)},
    "bad_sync": {"whole": (2, 2048, 2048), "whole_packed": (2, 2048, 2048, 2048), "block_loop": (2, 2048, 2048, 2048),
        "block_loop_readahead": (2, 2048, 2048, 2048), "resident_host": (2, 2048, 2048),
        "resident_device": (2, 2048, 2048), "files_resident": (2, 2, 0, 2048, 2048), "files_packed": (2, 2, 0),
        "index_host": (2, 2), "index_device": (2, 2)},
    "cut_in_size": {"whole": (4, 2048, 2048), "whole_packed": (4, 2048, 2048, 2048),
        "block_loop": (4, 2048, 2048, 2048), "block_loop_readahead": (4, 2048, 2048, 2048),
        "resident_host": (4, 2048, 2048), "resident_device": (4, 2048, 2048), "files_resident": (4, 4, 0, 2048, 2048),
        "files_packed": (4, 4, 0), "index_host": (4, 2), "index_device": (4, 2)},
    "cut_in_payload": {"whole": (4, 2048, 2048), "whole_packed": (4, 2048, 2048, 2048),
        "block_loop": (4, 2048, 2048, 2048), "block_loop_readahead": (4, 2048, 2048, 2048),
        "resident_host": (4, 2048, 2048), "resident_device": (4, 2048, 2048), "files_resident": (4, 4, 0, 2048, 2048),
        "files_packed": (4, 4, 0), "index_host": (4, 2), "index_device": (4, 2)},
    "size_below_5": {"whole": (2, 2048, 2048), "whole_packed": (2, 2048, 2048, 2048),
        "block_loop": (2, 2048, 2048, 2048), "block_loop_readahead": (2, 2048, 2048, 2048),
        "resident_host": (2, 2048, 2048), "resident_device": (2, 2048, 2048), "files_resident": (2, 2, 0, 2048, 2048),
        "files_packed": (2, 2, 0), "index_host": (2, 2), "index_device": (2, 2)},
    "type9_crc_on": {"whole": (6, 2048, 2048), "whole_packed": (6, 2048, 2048, 2048),
        "block_loop": (6, 2048, 2048, 2048), "block_loop_readahead": (6, 2048, 2048, 2048),
        "resident_host": (6, 2048, 2048), "resident_device": (6, 2048, 2048), "files_resident": (6, 6, 0, 2048, 2048),
        "files_packed": (6, 6, 0), "index_host": (2, 2), "index_device": (2, 2)},
    "type9_crc_off": {"whole": (2, 2048, 2048), "whole_packed": (2, 2048, 2048, 2048),
        "block_loop": (2, 2048, 2048, 2048), "block_loop_readahead": (2, 2048, 2048, 2048),
        "resident_host": (2, 2048, 2048), "resident_device": (2, 2048, 2048), "files_resident": (2, 2, 0, 2048, 2048),
        "files_packed": (2, 2, 0), "index_host": (2, 2), "index_device": (2, 2)},
    "raw_cut": {"whole": (4, 3072, 3072), "whole_packed": (4, 3072, 3072, 3072), "block_loop": (4, 3072, 3072, 3072),
        "block_loop_readahead": (4, 3072, 3072, 3072), "resident_host": (4, 3072, 3072),
        "resident_device": (4, 3072, 3072), "files_resident": (4, 4, 0, 3072, 3072), "files_packed": (4, 4, 0),
        "index_host": (4, 3), "index_device": (4, 3)},
    "too_many_samples": {"whole": (3, 2048, 2048), "whole_packed": (3, 2048, 2048, 2048),
        "block_loop": (3, 2048, 2048, 2048), "block_loop_readahead": (3, 2048, 2048, 2048),
        "resident_host": (3, 2048, 2048), "resident_device": (3, 2048, 2048), "files_resident": (3, 3, 0, 2048, 2048),
        "files_packed": (3, 3, 0), "index_host": (3, 2), "index_device": (3, 2)},
    "crc_mismatch": {"whole": (6, 2048, 2048), "whole_packed": (6, 2048, 2048, 2048),
        "block_loop": (6, 2048, 2048, 2048), "block_loop_readahead": (6, 2048, 2048, 2048),
        "resident_host": (6, 2048, 6444), "resident_device": (6, 2048, 6444), "files_resident": (6, 6, 0, 2048, 6444),
        "files_packed": (6, 6, 0), "index_host": (0, 7), "index_device": (0, 7)},
    "ends_on_boundary": {"whole": (0, 4096, 4096), "whole_packed": (0, 4096, 4096, 4096),
        "block_loop": (0, 4096, 4096, 4096), "block_loop_readahead": (0, 4096, 4096, 4096),
        "resident_host": (0, 4096, 4096), "resident_device": (0, 4096, 4096), "files_resident": (0, 0, 0, 4096, 4096),
        "files_packed": (0, 0, 0), "index_host": (0, 4), "index_device": (0, 4)},
}


def run_case(codec, Mem, oracle, case):
    pcm, good = source(oracle)
    data, size, crc = damaged(oracle, good, case)
    img = padded(data)
    good_index = np.array([[k * BLOCK, off] for k, off in enumerate(block_offsets(good))], np.uint32)
    got = {}
    for name in ENTRY_POINTS:
        if name.startswith("index"):
            got[name] = index(codec, Mem, img, size, crc, pcm, good_index, name == "index_device")
        elif name.startswith("files"):
            got[name] = globals()["run_" + name](codec, Mem, img, size, crc, pcm, good)
        else:
            got[name] = globals()["run_" + name](codec, Mem, img, size, crc, pcm)
    return got


def check_case(codec, Mem, oracle, case):
    got = run_case(codec, Mem, oracle, case)
    want = EXPECTED[case]
    assert {k: tuple(v) for k, v in got.items()} == want


def silent_stream(oracle, blocks, block):
    pcm = np.zeros((2, blocks * block), np.int32)
    data = oracle.encode(pcm, preset=0, block=block)
    assert len(data) == 30 + 11 * blocks
    return pcm, data


def check_silent(codec, Mem, oracle, blocks, block):
    """every block of these streams is 11 bytes: the block table must not be sized from the byte count"""
    pcm, data = silent_stream(oracle, blocks, block)
    n = pcm.shape[1]
    img = padded(data)
    with Decoder(codec, 1) as d:
        raw = np.full(n * 4 + 64, PACKED_SENTINEL, np.uint8)
        files = (FileDesc * 1)(FileDesc(0, n, 0, len(data), 99))
        assert d.L.LINNEB200_DecodeFilesPacked(d.h, u8(img), len(data), files, 1, u8(raw)) == OK
        assert files[0].status == OK
        assert np.array_equal(packed_planes(raw, n, 2), pcm) and np.all(raw[n * 4:] == PACKED_SENTINEL)

        d_img = Mem(img)
        d_pcm = Mem(np.full((2, n + 4), SENTINEL, np.int32))
        files = (FileDesc * 1)(FileDesc(0, n, 0, len(data), 99))
        assert d.L.LINNEB200_DecodeFilesResident(d.h, C.c_void_p(d_img.ptr), len(data), files, 1, C.c_void_p(d_pcm.ptr), n + 4) == OK
        out = d_pcm.get()
        assert files[0].status == OK and np.array_equal(out[:, :n], pcm) and np.all(out[:, n:] == SENTINEL)

        d_pcm = Mem(np.full((2, n + 4), SENTINEL, np.int32))
        assert d.L.LINNEB200_DecodeWholeResident(d.h, None, C.c_void_p(d_img.ptr), len(data), C.c_void_p(d_pcm.ptr), n + 4, 2, n) == OK
        out = d_pcm.get()
        assert np.array_equal(out[:, :n], pcm) and np.all(out[:, n:] == SENTINEL)


CASES = ["intact", "bad_sync", "cut_in_size", "cut_in_payload", "size_below_5", "type9_crc_on", "type9_crc_off", "raw_cut",
         "too_many_samples", "crc_mismatch", "ends_on_boundary"]
SILENT = [(150, 1024), (600, 128)]


# ---- the simulator -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_framing_matrix_hostsim(hostsim, oracle, case):
    check_case(hostsim, HostMem, oracle, case)


@pytest.mark.parametrize("blocks,block", SILENT)
def test_silent_streams_hostsim(hostsim, oracle, blocks, block):
    check_silent(hostsim, HostMem, oracle, blocks, block)


# ---- the product ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_framing_matrix_gpu(gpu, oracle, case):
    check_case(gpu, CudaMem, oracle, case)


@pytest.mark.gpu
@pytest.mark.parametrize("blocks,block", SILENT)
def test_silent_streams_gpu(gpu, oracle, blocks, block):
    check_silent(gpu, CudaMem, oracle, blocks, block)
