"""window_bench.py -- random access on a long stream: seek-index build and sample-window decodes.

The stream is the BASELINE C3 shape: one hour of seeded synthetic 44.1 kHz 16-bit stereo at -m 7, block size 10240,
built with the GPU encoder.  Measured, in one run:
  - LINNEB200_DecoderBuildIndex on the host image and on the device image;
  - LINNEB200_DecodeWindows (host image in, host planes out), LINNEB200_DecodeWindowsPacked (host image in, packed
    WAV data-chunk bytes out, into a page-locked buffer) and LINNEB200_DecodeWindowsResident (both in HBM) for W
    one-second windows at seeded random starts, W in {1, 8, 64, 512, 4096};
  - DecodeWhole / DecodeWholePacked / DecodeWholeResident of the same stream, for comparison.
Every window of every W is checked against the slice of a whole-stream decode (the packed windows against the bytes of
DecodeWholePacked) before any time is reported.  Times are
medians of synchronous calls (host wall clock) after a warm-up.  One JSON line goes to stdout and to --out, with the GPU's
name and power limit read in the same run.

    python tools/window_bench.py [--seconds 3600] [--reps 7] [--out profiles/r4_windows_packed.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

RATE, BITS, BLOCK, PRESET = 44100, 16, 10240, 7
WINDOW_COUNTS = (1, 8, 64, 512, 4096)


def gpu_identity():
    """name and power limit of GPU 0 (read-only query)"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(",")]
        return name, limit
    except Exception as e:                                           # the numbers stay usable without it
        return f"unknown ({e})", "unknown"


def median_ms(fn, reps):
    fn()                                                             # warm-up: grows the handle's buffers
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(times))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_windows_packed.json"))
    args = ap.parse_args()

    import torch
    import harness
    from linne_b200 import EncoderSession, DecoderSession, SeekPoint, Window, OK
    if not torch.cuda.is_available():
        raise SystemExit("window_bench needs a CUDA device")
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
    d_stream[size:size + 64].zero_()
    h_stream = torch.zeros(size + 16, dtype=torch.uint8).pin_memory()
    h_stream[:size].copy_(d_stream[:size])
    u8p = C.POINTER(C.c_uint8)
    h_data = C.cast(h_stream.data_ptr(), u8p)

    dec = DecoderSession(channels=nch)
    L = dec.lib

    # ---- whole-stream decodes: the reference the windows are checked against, and the comparison ----
    h_full = torch.zeros((nch, n), dtype=torch.int32).pin_memory()
    full_ptrs = (C.POINTER(C.c_int32) * nch)(*[C.cast(h_full[c].data_ptr(), C.POINTER(C.c_int32)) for c in range(nch)])
    d_full = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    ms_whole = median_ms(lambda: dec.decode_whole(h_stream.data_ptr(), size, full_ptrs, nch, n), args.reps)
    ms_whole_res = median_ms(lambda: dec.decode_whole_resident(h_stream.data_ptr(), d_stream.data_ptr(), size,
                                                               d_full.data_ptr(), stride, nch, n), args.reps)
    frame = nch * BITS // 8
    h_full_pk = torch.zeros(n * frame, dtype=torch.uint8).pin_memory()
    frames = C.c_uint32(0)

    def whole_packed():
        rc = L.LINNEB200_DecodeWholePacked(dec.h, h_data, size, C.cast(h_full_pk.data_ptr(), u8p), n, C.byref(frames))
        assert rc == OK and frames.value == n, rc
    ms_whole_pk = median_ms(whole_packed, args.reps)
    full = h_full.numpy()
    full_pk = h_full_pk.numpy()
    assert np.array_equal(full, pcm), "whole-stream decode differs from the input"
    assert full_pk.tobytes() == harness.pack_pcm(pcm, BITS), "packed whole-stream decode differs from the input"
    assert torch.equal(d_full[:, :n], d_pcm[:, :n]), "resident whole-stream decode differs from the input"

    # ---- seek index, host hop and device hop ----
    count = C.c_uint32(0)
    assert L.LINNEB200_DecoderBuildIndex(dec.h, h_data, None, size, None, 0, C.byref(count)) in (OK, 3)
    N = count.value
    pts_host, pts_dev = (SeekPoint * N)(), (SeekPoint * N)()

    def index_host():
        rc = L.LINNEB200_DecoderBuildIndex(dec.h, h_data, None, size, pts_host, N, C.byref(count))
        assert rc == OK and count.value == N, rc

    def index_dev():
        rc = L.LINNEB200_DecoderBuildIndex(dec.h, None, C.c_void_p(d_stream.data_ptr()), size, pts_dev, N, C.byref(count))
        assert rc == OK and count.value == N, rc
    ms_index_host = median_ms(index_host, args.reps)
    ms_index_dev = median_ms(index_dev, args.reps)
    assert bytes(pts_host) == bytes(pts_dev), "host and device index differ"

    # ---- windows ----
    rng = np.random.default_rng(args.seed)
    results = {}
    for W in WINDOW_COUNTS:
        starts = rng.integers(0, n - RATE + 1, W)
        wins = (Window * W)(*[Window(int(s), RATE, w * RATE, 0) for w, s in enumerate(starts)])
        room = W * RATE
        out_t = torch.full((nch, room), -1, dtype=torch.int32).pin_memory()   # page-locked, as the whole decode's planes
        out = out_t.numpy()
        out_ptrs = (C.POINTER(C.c_int32) * nch)(*[out[c].ctypes.data_as(C.POINTER(C.c_int32)) for c in range(nch)])
        d_out = torch.full((nch, room), -1, dtype=torch.int32, device=dev)
        out_pk_t = torch.full((room * frame,), 0xA5, dtype=torch.uint8).pin_memory()
        out_pk = out_pk_t.numpy()

        def host_call():
            rc = L.LINNEB200_DecodeWindows(dec.h, h_data, size, pts_host, N, wins, W, out_ptrs, nch, room)
            assert rc == OK, rc

        def packed_call():
            rc = L.LINNEB200_DecodeWindowsPacked(dec.h, h_data, size, pts_host, N, wins, W, out_pk.ctypes.data_as(u8p), room)
            assert rc == OK, rc

        def resident_call():
            rc = L.LINNEB200_DecodeWindowsResident(dec.h, C.c_void_p(d_stream.data_ptr()), size, pts_host, N, wins, W,
                                                   C.c_void_p(d_out.data_ptr()), room)
            assert rc == OK, rc
        host_call()
        packed_call()
        resident_call()
        back = d_out.cpu().numpy()
        for w, s in enumerate(starts):
            want = full[:, s:s + RATE]
            assert np.array_equal(out[:, w * RATE:(w + 1) * RATE], want), f"W={W}: window {w} differs (host buffers)"
            assert np.array_equal(back[:, w * RATE:(w + 1) * RATE], want), f"W={W}: window {w} differs (resident)"
            assert np.array_equal(out_pk[w * RATE * frame:(w + 1) * RATE * frame], full_pk[s * frame:(s + RATE) * frame]), \
                f"W={W}: window {w} differs (packed)"
        marks = np.zeros(N + 1, np.int64)
        firsts = np.frombuffer(bytes(pts_host), np.uint32).reshape(-1, 2)[:, 0]
        k0 = np.searchsorted(firsts, starts, side="right") - 1
        k1 = np.searchsorted(firsts, starts + RATE - 1, side="right") - 1
        np.add.at(marks, k0, 1)
        np.add.at(marks, k1 + 1, -1)
        blocks = int(np.count_nonzero(np.cumsum(marks)[:N]))
        before = dec.launch_count()
        resident_call()
        launches = dec.launch_count() - before
        results[str(W)] = {"blocks": blocks, "launches": int(launches),
                           "host_ms": round(median_ms(host_call, args.reps), 3),
                           "packed_ms": round(median_ms(packed_call, args.reps), 3),
                           "resident_ms": round(median_ms(resident_call, args.reps), 3)}
    dec.close()

    def crossover(key, whole):
        return next((int(W) for W, r in results.items() if r[key] >= whole), None)

    line = {
        "workload": f"random access: {args.seconds:.0f} s 44.1 kHz 16-bit stereo, -m {PRESET}, block {BLOCK}, {N} blocks, "
                    f"{size} bytes; one-second windows at seeded random starts",
        "gpu": gpu_name, "power_limit": power_limit,
        "index_ms": {"host": round(ms_index_host, 3), "device": round(ms_index_dev, 3)},
        "whole_ms": {"host": round(ms_whole, 3), "packed": round(ms_whole_pk, 3), "resident": round(ms_whole_res, 3)},
        "windows": results,
        "first_W_not_faster_than_whole": {"host": crossover("host_ms", ms_whole), "packed": crossover("packed_ms", ms_whole_pk),
                                          "resident": crossover("resident_ms", ms_whole_res)},
        "checked": "every window equals the whole-stream decode slice (host planes and resident) or the DecodeWholePacked "
                   "bytes (packed)",
        "timing": f"median of {args.reps} synchronous calls after one warm-up, host wall clock",
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
