"""Pin the oracle (oracle/linne_oracle.c) to the reference: known-answer vectors from the reference's
own tests, the committed golden streams, and byte-for-byte comparison with the unmodified reference: live where
oracle/_ref was built, otherwise with the reference's answers stored in tests/golden/reference_record.json."""
import numpy as np
import pytest

import harness

# CRC16 known answers: reference test/linne_internal/main.cpp:25-32
CRC_KATS = [(bytes([0x00, 0x00, 0x00, 0x01]), 0xC0C1), (bytes([0x10, 0x00, 0x00, 0x00]), 0xC004),
            (bytes([0x00, 0xFF, 0xFF, 0x00]), 0xC071), (bytes([0xDE, 0xAD, 0xBE, 0xAF]), 0x159A),
            (bytes([0xAB, 0xAD, 0xCA, 0xFE]), 0xE566), (bytes([0x12, 0x34, 0x56, 0x78]), 0x347B)]


def test_crc16_known_answers(oracle):
    for data, want in CRC_KATS:
        assert oracle.crc16(data) == want


def test_huffman_known_answers(oracle):
    # reference test/static_huffman/main.cpp:40-73
    codes, lens = oracle.huffman_codes([4, 3, 2, 1])
    assert list(zip(codes, lens)) == [(0x0, 1), (0x2, 2), (0x7, 3), (0x6, 3)]
    codes, lens = oracle.huffman_codes([5, 3, 2, 1, 1])
    assert list(zip(codes, lens)) == [(0x0, 1), (0x2, 2), (0x6, 3), (0xE, 4), (0xF, 4)]
    # total code length checks, main.cpp:86-89
    for counts, total in (([8, 4, 4, 4, 2, 2], 60), ([50, 20, 10, 8, 5, 4, 2, 1], 220)):
        _, lens = oracle.huffman_codes(counts)
        assert int(np.sum(np.array(counts) * lens)) == total


def test_coef_code_lengths(oracle):
    _, lens = oracle.coef_table()
    assert lens.min() == 5 and lens.max() == 14 and lens[0] == 5       # SURVEY Appendix B


def test_rice_parameter_steps(oracle):
    # step positions probed on the reference formula (SURVEY Appendix B)
    for mean, k2 in ((0.0, 0), (2.5, 0), (2.53, 1), (5.6, 2), (11.5, 3), (95.4, 6), (191.2, 7), (382.8, 8)):
        assert oracle.rice_k2(mean) == k2


@pytest.mark.parametrize("name", harness.GOLDEN_CASES + ["mixed_types_m5"])
def test_golden_streams(oracle, name):
    g = harness.load_golden(name)
    pcm, stream = g["pcm"], g["stream"].tobytes()
    assert np.array_equal(oracle.decode(stream), pcm)
    assert oracle.encode(pcm, bits=int(g["bits"]), block=int(g["block"]), preset=int(g["preset"])) == stream


# ---- comparison with the unmodified reference: live where oracle/_ref was built, else with its stored answers ----
def test_live_crc_and_huffman(oracle, reference):
    rng = np.random.default_rng(3)
    for n in (1, 7, 64, 1000, 40971):
        data = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        assert oracle.crc16(data) == reference.expect(f"crc16/{n}", lambda r: r.crc16(data))
    for i, counts in enumerate(([1, 1, 1, 1], [0, 5, 0, 9, 2], list(rng.integers(0, 1000, 200)))):
        ours = [a.tolist() for a in oracle.huffman_codes(counts)]
        assert ours == reference.expect(f"huffman/{i}", lambda r: [a.tolist() for a in r.huffman_codes(counts)])


def _encode_identical(oracle, reference, key, pcm, **kw):
    """oracle.encode(pcm, **kw) gives the reference's bytes, and decodes back to pcm."""
    ours = oracle.encode(pcm, **kw)
    assert harness.digest(ours) == reference.expect(key, lambda r: harness.digest(r.encode(pcm, **kw))), key
    assert np.array_equal(oracle.decode(ours), pcm), key


@pytest.mark.parametrize("preset", range(8))
def test_live_streams_identical(oracle, reference, preset):
    pcm = harness.synth_pcm(seconds=1.2, channels=2, bits=16, seed=40 + preset)
    _encode_identical(oracle, reference, f"streams/m{preset}", pcm, preset=preset)


@pytest.mark.parametrize("channels,bits", [(1, 8), (2, 24), (8, 24), (3, 16)])
def test_live_formats_identical(oracle, reference, channels, bits):
    pcm = harness.synth_pcm(n=2600, channels=channels, bits=bits, seed=7)
    for preset in (0, 5):
        _encode_identical(oracle, reference, f"formats/{channels}ch{bits}/m{preset}", pcm, bits=bits, preset=preset, block=1024)


def test_live_reference_generators_roundtrip(oracle, reference):
    # the nine generators of test/linne_encode_decode/main.cpp at 8192 samples / block 1024
    for name, gen in harness.reference_test_generators().items():
        for channels, bits, preset in ((1, 16, 0), (2, 8, 7), (2, 24, 7)):
            pcm = harness.to_fixed(gen(channels, 8192), bits)
            _encode_identical(oracle, reference, f"generators/{name}/{channels}ch{bits}/m{preset}", pcm,
                              bits=bits, rate=8000, block=1024, preset=preset)


def test_live_af_and_learning_identical(oracle, reference):
    pcm = harness.synth_pcm(n=2048, channels=1, bits=16, seed=9)
    _encode_identical(oracle, reference, "af2", pcm, preset=0, block=1024, af=2)
    _encode_identical(oracle, reference, "learning1", pcm[:, :1024], preset=0, block=1024, learning=1)
