"""Generate tests/golden/*.npz with the UNMODIFIED reference (oracle/_ref/liblinne_ref.so, built from its sources
by `make -C oracle ref REF=<reference checkout>`):  python tests/golden/make_golden.py

Each fixture holds the PCM, the reference's .lnn bytes and, per compressed block-channel, the
analysis results the reference kept in its handle (unit counts, shifts, quantised coefficients,
pre-emphasis state) plus the residual -- so the parity tests can check
  * oracle / GPU decode(reference bytes) == PCM                       (bit-exact decode)
  * oracle encode == reference bytes                                   (oracle pinned)
  * GPU pack(reference coefficients) == reference bytes                (identical coefficients -> identical bits)
without the reference being present.

    python tests/golden/make_golden.py --record    writes tests/golden/reference_record.json instead: the answers
the comparison tests of test_oracle_vs_reference.py and test_cli.py ask of the reference (CRCs, Huffman tables,
stream digests), taken by running those tests with a recording harness.ReferenceRecord.  They come from
oracle/_ref where it was built; otherwise from the oracle, which those same tests pin to the reference byte for
byte wherever oracle/_ref exists (they then check every stored answer against the live reference).  The file names
its source.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import harness  # noqa: E402

CASES = [
    # name, channels, bits, samples, block, preset, seed
    ("stereo16_m0", 2, 16, 5000, 2048, 0, 21),
    ("stereo16_m4", 2, 16, 5000, 2048, 4, 22),
    ("stereo16_m7", 2, 16, 5000, 2048, 7, 23),
    ("mono8_m7", 1, 8, 3000, 1024, 7, 24),
    ("eightch24_m7", 8, 24, 2304, 1024, 7, 25),
    ("mono24_m2", 1, 24, 4096, 4096, 2, 26),
]


def record():
    import test_cli
    import test_oracle_vs_reference as t
    oracle = harness.Oracle()
    live, source = (harness.Ref(), "reference") if harness.have_ref() else (oracle, "oracle")
    rec = harness.ReferenceRecord(live, recording=True)
    t.test_live_crc_and_huffman(oracle, rec)
    for preset in range(8):
        t.test_live_streams_identical(oracle, rec, preset)
    for channels, bits in [(1, 8), (2, 24), (8, 24), (3, 16)]:
        t.test_live_formats_identical(oracle, rec, channels, bits)
    t.test_live_reference_generators_roundtrip(oracle, rec)
    t.test_live_af_and_learning_identical(oracle, rec)
    for case in test_cli.CASES:
        test_cli.reference_cli_answer(rec, case)
    with open(harness.RECORD_JSON, "w") as f:
        json.dump({"source": source, "answers": rec.answers}, f, indent=0, sort_keys=True)
        f.write("\n")
    print(harness.RECORD_JSON, len(rec.answers), "answers from the", source)


def main():
    ref = harness.Ref()
    for name, ch, bits, n, block, preset, seed in CASES:
        pcm = harness.synth_pcm(n=n, channels=ch, bits=bits, seed=seed)
        stream, blocks = ref.encode_blocks_traced(pcm, bits=bits, block=block, preset=preset)
        assert np.array_equal(ref.decode(stream), pcm)
        layers = harness.PRESET_LAYERS[preset]
        nb = len(blocks)
        units = np.zeros((nb, ch, 3), np.uint8); rshift = np.zeros((nb, ch, 3), np.uint8)
        coef = np.zeros((nb, ch, 3, 128), np.int8)
        preem_prev = np.zeros((nb, ch, 2), np.int32); preem_coef = np.zeros((nb, ch, 2), np.uint8)
        types = np.array([b["type"] for b in blocks], np.uint8)
        for bi, b in enumerate(blocks):
            for c, chd in enumerate(b["channels"]):
                for l, P in enumerate(layers):
                    units[bi, c, l] = chd["units"][l]; rshift[bi, c, l] = chd["rshift"][l]
                    coef[bi, c, l, :P] = chd["coef"][l]
                preem_prev[bi, c] = chd["preem_prev"]; preem_coef[bi, c] = chd["preem_coef"]
        np.savez_compressed(os.path.join(HERE, name + ".npz"), pcm=pcm.astype(np.int32),
                            stream=np.frombuffer(stream, np.uint8), bits=bits, block=block, preset=preset,
                            types=types, units=units, rshift=rshift, coef=coef,
                            preem_prev=preem_prev, preem_coef=preem_coef)
        print(name, len(stream), "bytes", nb, "blocks")
    # the three block types in one stream
    pcm = harness.mixed_types_pcm(sr=8192)
    stream = ref.encode(pcm, preset=5, block=2048)
    assert np.array_equal(ref.decode(stream), pcm)
    np.savez_compressed(os.path.join(HERE, "mixed_types_m5.npz"), pcm=pcm, stream=np.frombuffer(stream, np.uint8),
                        bits=16, block=2048, preset=5)
    print("mixed_types_m5", len(stream))


if __name__ == "__main__":
    record() if sys.argv[1:] == ["--record"] else main()
