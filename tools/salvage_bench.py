"""salvage_bench.py -- salvage decodes of a long stream, intact and damaged, against the whole-stream decodes.

The stream is the BASELINE C3 shape: one hour of seeded synthetic 44.1 kHz 16-bit stereo at -m 7, block size 10240,
built with the GPU encoder (as tools/window_bench.py builds it).  Measured, in one run:
  - LINNEB200_DecodeSalvage / DecodeSalvagePacked on the intact stream, and DecodeWhole / DecodeWholePacked;
  - both salvage calls on the stream with 1, 16 and 256 seeded payload bit flips (each in its own compressed block) and
    with one framing gap (the sync code of the middle block flipped);
  - the device time of the resynchronising scan and of the candidates' CRC pass (per-stage CUDA events, in a pass of its
    own after the timed ones).
Every salvage output is checked before any time is reported: on the intact stream it must equal the whole-stream decode
byte for byte; on a damaged one every sample outside the reported records must equal the input and every sample inside
must be zero.  Times are medians of synchronous calls (host wall clock, host buffers in and out) after a warm-up.  One
JSON line goes to stdout and to --out, with the GPU's name and power limit read in the same run.

    python tools/salvage_bench.py [--seconds 3600] [--reps 7] [--out profiles/r5_salvage.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

from window_bench import RATE, BITS, BLOCK, PRESET, gpu_identity, median_ms   # noqa: E402

FLIPS = (1, 16, 256)


def block_table(data):
    """(byte offset, byte size, type) of every block of an intact stream"""
    off, out = 30, []
    while off < len(data):
        size = int.from_bytes(data[off + 2:off + 6], "big") + 6
        out.append((off, size, data[off + 8]))
        off += size
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_salvage.json"))
    args = ap.parse_args()

    import torch
    import harness
    from linne_b200 import EncoderSession, DecoderSession, Damage, LINNEHeader, OK, DATA_CORRUPTION
    if not torch.cuda.is_available():
        raise SystemExit("salvage_bench needs a CUDA device")
    dev = torch.device("cuda:0")
    gpu_name, power_limit = gpu_identity()

    # ---- the stream: a seeded 30 s clip repeated to the length asked for, encoded on the GPU ----
    clip = harness.synth_pcm(seconds=30.0, sr=RATE, channels=2, bits=BITS, seed=args.seed)
    n = int(round(args.seconds * RATE))
    pcm = np.ascontiguousarray(np.tile(clip, (1, (n + clip.shape[1] - 1) // clip.shape[1]))[:, :n])
    nch = pcm.shape[0]
    stride = (n + 4 + 3) // 4 * 4
    d_pcm = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    d_pcm[:, :n].copy_(torch.from_numpy(pcm))
    cap = 30 + nch * n * 2 + 11 * (n // BLOCK + 2) + 65536
    d_stream = torch.zeros(cap + 64, dtype=torch.uint8, device=dev)
    enc = EncoderSession(nch, bits=BITS, rate=RATE, block=BLOCK, preset=PRESET)
    size = enc.encode_whole_resident(d_pcm.data_ptr(), stride, n, d_stream.data_ptr(), cap)
    enc.close()
    good = d_stream[:size].cpu().numpy().tobytes()
    del d_stream, d_pcm
    blocks = block_table(good)

    dec = DecoderSession(channels=nch)
    L = dec.lib
    u8p = C.POINTER(C.c_uint8)
    hdr = LINNEHeader()
    h_img = torch.zeros(size + 16, dtype=torch.uint8).pin_memory()
    h_img_np = h_img.numpy()
    h_img_np[:size] = np.frombuffer(good, np.uint8)
    img_ptr = C.cast(h_img.data_ptr(), u8p)
    assert L.LINNEDecoder_DecodeHeader(img_ptr, size, C.byref(hdr)) == OK
    assert L.LINNEDecoder_SetHeader(dec.h, C.byref(hdr)) == OK

    h_planes = torch.zeros((nch, n), dtype=torch.int32).pin_memory()
    planes_ptrs = (C.POINTER(C.c_int32) * nch)(*[C.cast(h_planes[c].data_ptr(), C.POINTER(C.c_int32)) for c in range(nch)])
    frame = nch * BITS // 8
    h_packed = torch.zeros(n * frame, dtype=torch.uint8).pin_memory()
    packed_ptr = C.cast(h_packed.data_ptr(), u8p)
    damage = (Damage * 1024)()
    count = C.c_uint32(0)
    frames = C.c_uint32(0)

    def whole():
        assert L.LINNEDecoder_DecodeWhole(dec.h, img_ptr, size, planes_ptrs, nch, n) == OK

    def whole_packed():
        assert L.LINNEB200_DecodeWholePacked(dec.h, img_ptr, size, packed_ptr, n, C.byref(frames)) == OK

    def salvage(data_size, want):
        def call():
            assert L.LINNEB200_DecodeSalvage(dec.h, img_ptr, data_size, planes_ptrs, nch, n, damage, 1024, C.byref(count)) == want
        return call

    def salvage_packed(data_size, want):
        def call():
            assert L.LINNEB200_DecodeSalvagePacked(dec.h, img_ptr, data_size, packed_ptr, n, damage, 1024, C.byref(count)) == want
        return call

    def records():
        return [(d.first_sample, d.num_samples, d.byte_offset, d.byte_size, d.status) for d in damage[:count.value]]

    def check(recs):
        lost = np.zeros(n, bool)
        for s, k, _, _, _ in recs:
            lost[s:s + k] = True
        got = h_planes.numpy()
        assert np.array_equal(got[:, ~lost], pcm[:, ~lost]) and np.all(got[:, lost] == 0), "salvage output differs"
        assert h_packed.numpy().tobytes() == harness.pack_pcm(got, BITS), "packed salvage output differs from the planes"

    def load(data):
        h_img_np[:len(data)] = np.frombuffer(data, np.uint8)
        h_img_np[len(data):] = 0
        # the handle keeps the intact stream's header: a damaged image is read from byte 30 on
        assert L.LINNEDecoder_SetHeader(dec.h, C.byref(hdr)) == OK

    result = {"workload": f"{args.seconds:.0f} s 44.1 kHz 16-bit stereo, -m {PRESET}, block {BLOCK}",
              "stream_bytes": size, "blocks": len(blocks), "gpu": gpu_name, "power_limit": power_limit,
              "timing": f"median of {args.reps} synchronous calls after a warm-up, host buffers (page-locked)"}

    # ---- the intact stream ----
    load(good)
    result["decode_whole_ms"] = median_ms(whole, args.reps)
    assert np.array_equal(h_planes.numpy(), pcm)
    result["decode_whole_packed_ms"] = median_ms(whole_packed, args.reps)
    ref_packed = h_packed.numpy().tobytes()
    assert ref_packed == harness.pack_pcm(pcm, BITS)
    h_planes.zero_(); h_packed.zero_()
    result["salvage_intact_ms"] = median_ms(salvage(size, OK), args.reps)
    assert count.value == 0 and np.array_equal(h_planes.numpy(), pcm)
    result["salvage_packed_intact_ms"] = median_ms(salvage_packed(size, OK), args.reps)
    assert count.value == 0 and h_packed.numpy().tobytes() == ref_packed

    # ---- damaged streams ----
    rng = np.random.default_rng(args.seed)
    compressed = [k for k, (_, sz, t) in enumerate(blocks) if t == 0 and sz > 64]
    cases = {}
    for f in FLIPS:
        b = bytearray(good)
        for k in sorted(rng.choice(compressed, size=f, replace=False).tolist()):
            off, sz, _ = blocks[k]
            b[off + 11 + int(rng.integers(0, sz - 11))] ^= 1 << int(rng.integers(0, 8))
        cases[f"flips_{f}"] = bytes(b)
    b = bytearray(good)
    b[blocks[len(blocks) // 2][0]] ^= 0x01
    cases["framing_gap_1"] = bytes(b)
    result["damaged"] = {}
    for name, data in cases.items():
        load(data)
        ms = median_ms(salvage(len(data), DATA_CORRUPTION), args.reps)
        ms_pk = median_ms(salvage_packed(len(data), DATA_CORRUPTION), args.reps)
        recs = records()
        check(recs)
        result["damaged"][name] = {"salvage_ms": ms, "salvage_packed_ms": ms_pk, "records": len(recs),
                                   "lost_samples": int(sum(r[1] for r in recs))}

    # ---- device time of the scan and the CRC pass (profiled pass of its own) ----
    load(good)
    dec.set_profiling(True)
    dec.reset_stage_stats()
    for _ in range(args.reps):
        salvage(size, OK)()
    stats = dec.stage_stats()
    dec.set_profiling(False)
    result["stages_per_call_ms"] = {k: v[1] / args.reps for k, v in stats.items()}
    line = json.dumps(result)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
