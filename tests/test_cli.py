"""The batch command-line driver (tools/linne_b200_cli, SURVEY section 8f.1) against the reference's own tool
(tools/linne_codec/linne_codec.c built unmodified by oracle/Makefile into oracle/_ref/linne_ref):
same options, same WAV <-> .lnn mapping, several files per invocation.

CPU-only: the driver linked against the host simulator (exercises WAV parsing, option handling, EncodeWhole /
DecodeWhole plumbing).  GPU: the driver on liblinne_b200.so, and the UNMODIFIED reference tool linked against
liblinne_b200.so (oracle/_ref/linne_ref_b200) -- the drop-in boundary exercised by the reference's own caller."""
import os
import struct
import subprocess

import numpy as np
import pytest

import harness

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_CLI = os.path.join(ROOT, "oracle", "_ref", "linne_ref")
REF_CLI_B200 = os.path.join(ROOT, "oracle", "_ref", "linne_ref_b200")
HOSTSIM_CLI = os.path.join(ROOT, "tests", "hostsim", "linne_hostsim_cli")
B200_CLI = os.path.join(ROOT, "linne_b200", "linne_b200_cli")


def write_wav(path, pcm, bits, rate=44100):
    """pcm: int32 [C][n] right-justified."""
    nch, n = pcm.shape
    nbytes = bits // 8
    inter = pcm.T.reshape(-1).astype(np.int64)
    if bits == 8:
        data = ((inter + 128) & 0xFF).astype(np.uint8).tobytes()
    else:
        raw = (inter & ((1 << bits) - 1)).astype(np.uint64)
        data = b"".join(raw.astype("<u8").tobytes()[i * 8:i * 8 + nbytes] for i in range(len(raw))) if bits == 24 \
            else raw.astype("<u2").tobytes()
    hdr = b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVEfmt " + struct.pack(
        "<IHHIIHH", 16, 1, nch, rate, rate * nch * nbytes, nch * nbytes, bits) + b"data" + struct.pack("<I", len(data))
    with open(path, "wb") as f:
        f.write(hdr + data)


def wav_data(path):
    raw = open(path, "rb").read()
    i = raw.index(b"data")
    return raw[20:36], raw[i + 8:i + 8 + struct.unpack("<I", raw[i + 4:i + 8])[0]]


def run(*cmd):
    res = subprocess.run(list(cmd), capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, (cmd, res.stdout[-400:], res.stderr[-400:])
    return res


CASES = [(2, 16, 2, 10240 * 2 + 2048, 11), (1, 24, 5, 10240 + 4096, 12), (2, 8, 0, 10240, 13)]   # ch, bits, preset, frames, seed


def reference_cli_answer(reference, case):
    """Digest of the reference tool's .lnn for a CASES entry: the tool encodes with block 10240 and M/S for two or more
    channels (linne_codec.c), which is the reference library's EncodeWhole with the harness defaults."""
    ch, bits, preset, n, seed = case
    pcm = harness.synth_pcm(n=n, channels=ch, bits=bits, seed=seed)
    return reference.expect(f"cli/{seed}", lambda r: harness.digest(r.encode(pcm, bits=bits, rate=44100, block=10240, preset=preset)))


def roundtrip(cli, tmp_path, tag, reference):
    """Our tool's .lnn equals the reference tool's (run where it was built, else its stored digest) and decodes back."""
    live = os.path.exists(REF_CLI)
    outs = []
    for case in CASES:
        ch, bits, preset, n, seed = case
        pcm = harness.synth_pcm(n=n, channels=ch, bits=bits, seed=seed)
        wav = tmp_path / f"in_{tag}_{seed}.wav"
        write_wav(str(wav), pcm, bits)
        ref_lnn = tmp_path / f"ref_{tag}_{seed}.lnn"
        if live:
            run(REF_CLI, "-e", "-m", str(preset), str(wav), str(ref_lnn))
        outs.append((wav, ref_lnn, preset, tmp_path / f"our_{tag}_{seed}.lnn", tmp_path / f"our_{tag}_{seed}.wav",
                     reference_cli_answer(reference, case)))
    # several files per invocation, grouped by preset (one option set per run)
    for wav, ref_lnn, preset, our_lnn, our_wav, _ in outs:
        run(cli, "-e", "-m", str(preset), str(wav), str(our_lnn))
    pairs = tmp_path / f"pairs_{tag}.txt"
    pairs.write_text("".join(f"{o[3]} {o[4]}\n" for o in outs))
    run(cli, "-d", "-L", str(pairs))                               # list file, one handle for all
    for wav, ref_lnn, preset, our_lnn, our_wav, want in outs:
        assert harness.digest(our_lnn.read_bytes()) == want, f"stream differs from the reference tool's ({wav.name})"
        assert wav_data(str(our_wav)) == wav_data(str(wav))
        if live:
            assert our_lnn.read_bytes() == ref_lnn.read_bytes(), f"stream differs from the reference tool's ({wav.name})"
            ref_wav = tmp_path / ("back_" + ref_lnn.name + ".wav")
            run(REF_CLI, "-d", str(our_lnn), str(ref_wav))       # the reference tool decodes our file
            assert wav_data(str(ref_wav)) == wav_data(str(wav))


@pytest.mark.skipif(not os.path.exists(HOSTSIM_CLI), reason="CLI binary not built")
def test_cli_hostsim_matches_reference_tool(tmp_path, reference):
    roundtrip(HOSTSIM_CLI, tmp_path, "sim", reference)


def pipeline(cli, tmp_path, tag):
    """SURVEY 8f.3: many files through `-j N` workers give the files the one-worker run gives."""
    import json
    pairs_e, pairs_d, files = [], [], []
    for i in range(7):
        ch, bits, n = [(2, 16, 10240 + 512 * i), (1, 24, 4096 + 100 * i), (2, 8, 3000 + i)][i % 3]
        pcm = harness.synth_pcm(n=n, channels=ch, bits=bits, seed=40 + i)
        wav = tmp_path / f"p_{tag}_{i}.wav"
        write_wav(str(wav), pcm, bits)
        files.append((wav, tmp_path / f"p_{tag}_{i}.j1.lnn", tmp_path / f"p_{tag}_{i}.j3.lnn", tmp_path / f"p_{tag}_{i}.back.wav"))
    for col, jobs in ((1, "1"), (2, "3")):
        lst = tmp_path / f"enc_{tag}_{jobs}.txt"
        lst.write_text("".join(f"{f[0]} {f[col]}\n" for f in files))
        res = run(cli, "-e", "-m", "2", "-j", jobs, "-s", "-L", str(lst))
        stats = json.loads(res.stderr.strip().splitlines()[-1])
        assert stats["files"] == len(files) and stats["workers"] == int(jobs) and stats["samples"] > 0
    lst = tmp_path / f"dec_{tag}.txt"
    lst.write_text("".join(f"{f[2]} {f[3]}\n" for f in files))
    run(cli, "-d", "-j", "3", "-L", str(lst))
    for wav, one, three, back in files:
        assert one.read_bytes() == three.read_bytes()
        assert wav_data(str(back)) == wav_data(str(wav))
    # a missing file fails that pair only; the others are still written
    lst = tmp_path / f"bad_{tag}.txt"
    good = tmp_path / f"good_{tag}.lnn"
    lst.write_text(f"{tmp_path / 'nope.wav'} {tmp_path / 'nope.lnn'}\n{files[0][0]} {good}\n")
    res = subprocess.run([cli, "-e", "-m", "2", "-j", "2", "-L", str(lst)], capture_output=True, text=True, timeout=600)
    assert res.returncode != 0 and good.read_bytes() == files[0][1].read_bytes()


@pytest.mark.skipif(not os.path.exists(HOSTSIM_CLI), reason="CLI binary not built")
def test_cli_hostsim_file_pipeline(tmp_path):
    pipeline(HOSTSIM_CLI, tmp_path, "sim")


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(B200_CLI), reason="CLI binary not built")
def test_cli_b200_file_pipeline(tmp_path):
    pipeline(B200_CLI, tmp_path, "gpu")


@pytest.mark.skipif(not os.path.exists(HOSTSIM_CLI), reason="CLI binary not built")
def test_cli_usage_errors(tmp_path):
    for args in (["-e"], ["-e", "-d", "a", "b"], ["-e", "-m", "9", "a", "b"], ["-x", "a", "b"], ["-e", "only_one"]):
        assert subprocess.run([HOSTSIM_CLI] + args, capture_output=True).returncode != 0
    assert subprocess.run([HOSTSIM_CLI, "-e", str(tmp_path / "missing.wav"), str(tmp_path / "o.lnn")],
                          capture_output=True).returncode != 0


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(B200_CLI), reason="CLI binary not built")
def test_cli_b200_matches_reference_tool(tmp_path, reference):
    roundtrip(B200_CLI, tmp_path, "gpu", reference)


@pytest.mark.gpu
@pytest.mark.skipif(not (os.path.exists(REF_CLI) and os.path.exists(REF_CLI_B200)), reason="CLI binaries not built")
def test_unmodified_reference_tool_on_the_b200_library(tmp_path):
    """tools/linne_codec/linne_codec.c compiled as is, linked against liblinne_b200.so (INTEGRATION.md section 1)."""
    ch, bits, preset, n, seed = CASES[0]
    pcm = harness.synth_pcm(n=n, channels=ch, bits=bits, seed=seed)
    wav, a, b, back = (tmp_path / x for x in ("in.wav", "ref.lnn", "b200.lnn", "back.wav"))
    write_wav(str(wav), pcm, bits)
    run(REF_CLI, "-e", "-m", str(preset), str(wav), str(a))
    run(REF_CLI_B200, "-e", "-m", str(preset), str(wav), str(b))
    assert a.read_bytes() == b.read_bytes()
    run(REF_CLI_B200, "-d", str(a), str(back))
    assert wav_data(str(back)) == wav_data(str(wav))
