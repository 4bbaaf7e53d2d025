#!/usr/bin/env python
"""bench.py -- LINNE block encode/decode throughput on B200 (BASELINE.json metric).

Workload (BASELINE.json configs[1], "C2"): the synthetic 10 s / 44.1 kHz / 16-bit / stereo clip
(sinusoid mixture + coloured noise + transients, SURVEY Appendix B.1), encoded AND decoded at every
preset -m 0..7.  One step = the whole sweep: 8 x (EncodeWhole + DecodeWhole).  Samples are counted
once per preset (a sample that went through encode and decode counts once), so

    value [MSamples/s] = 8 presets x 882 000 samples x n_gpus / (ms_per_step / 1000) / 1e6.

  value : inputs resident in HBM (PCM planes and .lnn image on the device, LINNEB200_*Resident)
  e2e   : the reference-facing C-ABI with HOST buffers (pinned), H2D/D2H inside the timed region

Multi-GPU: blocks/files are independent, so ranks run the same sweep on their own copy of the clip
with no data-path collective ("weak"); time = max over ranks.

--impl reference times the unmodified reference (oracle/_ref/liblinne_ref.so, its own CPU code)
on the host cores, one thread per preset, same sweep.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

# Sixteen handles (8 encoders + 8 decoders) run on their own CUDA streams; with the default of 8 hardware
# work queues several streams share one queue and a kernel waiting for SMs blocks unrelated work behind it.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

CLIP_SECONDS, RATE, BITS, CHANNELS, BLOCK = 10.0, 44100, 16, 2, 10240
PRESETS = list(range(8))
# algorithmic MACs per input sample of the default analysis, per preset (SURVEY section 8a)
MAC_PER_SAMPLE = {0: 420, 1: 630, 2: 934, 3: 1401, 4: 2335, 5: 1802, 6: 2703, 7: 4505}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons while the timed region runs.  NVML in-process (one cheap call per sample); the
    nvidia-smi command line is only the fall-back: a new nvidia-smi process per rank every 200 ms initialises NVML for
    every GPU of the box and disturbed the timed region at 8 ranks."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()
        self.nvml = self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and all(x.strip().isdigit() for x in visible.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flag = lambda name: "Active" if r & getattr(n, name, 0) else "Not Active"
        return [str(sm), str(mx), flag("nvmlClocksThrottleReasonHwSlowdown"), flag("nvmlClocksThrottleReasonHwThermalSlowdown"),
                flag("nvmlClocksThrottleReasonSwThermalSlowdown"), flag("nvmlClocksThrottleReasonSwPowerCap")]

    def run(self):
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self.samples.append(self.sample_nvml())
                else:
                    out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    parts = [x.strip() for x in out.strip().split(",")]
                    if len(parts) >= 6:
                        self.samples.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.05 if self.nvml is not None else 0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i] == "Active" for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def make_clip():
    import harness
    return harness.synth_pcm(seconds=CLIP_SECONDS, sr=RATE, channels=CHANNELS, bits=BITS, seed=1)


DUMP_LIMIT_BYTES = 64_000_000        # all files --dump-outputs writes, together
DUMP_FRAMES = 1 << 17                # decoded frames kept per preset


def dump_outputs(path, streams, decoded):
    """--dump-outputs: what the last timed sweep step returned, as float32 .npy files, so that two builds can be compared
    file for file.  m<preset>_stream.npy is the whole compressed stream of that preset (one value per byte);
    m<preset>_decoded.npy is its decoded PCM [channel][frame] at DUMP_FRAMES frame positions drawn once with a fixed seed
    (sorted, the same for every preset and run): eight full planes would not fit the size limit beside the streams.
    The clip is 16-bit, so every value is exact in float32.  Should the streams leave less room than that, fewer frames
    are kept (with a warning on stderr), and nothing is written if the streams alone exceed the limit: the bench itself
    goes on either way."""
    arrays = {f"m{m}_stream": streams[m].cpu().numpy().astype(np.float32) for m in sorted(streams)}
    room = DUMP_LIMIT_BYTES - sum(a.nbytes for a in arrays.values()) - 2 * 128 * len(arrays)     # 128: an .npy header
    nch, n = next(iter(decoded.values())).shape
    if room < 0:
        print(f"bench.py: --dump-outputs writes nothing: the streams alone exceed {DUMP_LIMIT_BYTES} bytes", file=sys.stderr)
        return
    keep = min(n, DUMP_FRAMES, room // (4 * nch * len(decoded)))
    if keep < min(n, DUMP_FRAMES):
        print(f"bench.py: --dump-outputs keeps {keep} decoded frames per preset to stay within {DUMP_LIMIT_BYTES} bytes",
              file=sys.stderr)
    frames = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
    for m in sorted(decoded):
        arrays[f"m{m}_decoded"] = decoded[m].cpu().numpy()[:, frames].astype(np.float32)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# =================================================================================================
# reference arm
# =================================================================================================
def run_reference(args, rank, world):
    import harness
    if rank != 0:
        return
    if harness.have_ref():
        impl, kind = harness.Ref(), "reference"
    else:
        impl, kind = harness.Oracle(), "port"
    pcm = make_clip()
    n_samples = pcm.shape[0] * pcm.shape[1]
    ncpu = os.cpu_count() or 1
    # Blocks are independent (SURVEY Appendix B: a fresh handle per block reproduces EncodeWhole byte
    # for byte), so the fairest multi-core use of the single-threaded reference is one handle per
    # (preset, contiguous block range): tasks = 8 presets x `parts` ranges, run on all host cores.
    total_blocks = (pcm.shape[1] + BLOCK - 1) // BLOCK
    parts = max(1, min(total_blocks, ncpu // len(PRESETS)))
    per = (total_blocks + parts - 1) // parts
    ranges = [(b * BLOCK, min((b + per) * BLOCK, pcm.shape[1])) for b in range(0, total_blocks, per)]
    cores = min(ncpu, len(PRESETS) * len(ranges))

    def one_task(m, lo, hi, out):
        sub = np.ascontiguousarray(pcm[:, lo:hi])
        t0 = time.perf_counter(); s = impl.encode(sub, preset=m); t1 = time.perf_counter()
        d = impl.decode(s); t2 = time.perf_counter()
        out[(m, lo)] = (t1 - t0, t2 - t1, len(s) - 30, bool(np.array_equal(d, sub)))

    def sweep():
        res = {}
        pending = [(m, lo, hi) for m in PRESETS[::-1] for lo, hi in ranges]      # longest presets first
        lock = threading.Lock()

        def worker():
            while True:
                with lock:
                    if not pending:
                        return
                    m, lo, hi = pending.pop(0)
                one_task(m, lo, hi, res)
        threads = [threading.Thread(target=worker) for _ in range(cores)]
        t0 = time.perf_counter()
        for t in threads: t.start()
        for t in threads: t.join()
        per_preset = {}
        for (m, _), v in res.items():
            a = per_preset.setdefault(m, [0.0, 0.0, 30, True])
            a[0] += v[0]; a[1] += v[1]; a[2] += v[2]; a[3] = a[3] and v[3]
        return time.perf_counter() - t0, per_preset

    for _ in range(args.warmup):
        sweep()
    times, last = [], None
    for _ in range(args.steps):
        dt, last = sweep()
        times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = len(PRESETS) * n_samples / (ms / 1e3) / 1e6
    line = {
        "impl": "reference", "metric": "encode+decode MSamples/s over the -m 0..7 sweep", "value": round(value, 4),
        "unit": "MSamples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32+f64", "data": "synthetic",
        "config": {"workload": "C2: 10 s 44.1 kHz 16-bit stereo synthetic clip, -m 0..7 sweep, encode+decode",
                   "block": BLOCK, "ms": 1, "presets": PRESETS},
        "cpu_baseline": {"value": round(value, 4), "unit": "MSamples/s", "cores": cores, "kind": kind,
                         "sample": f"the full sweep (8 presets x 882000 samples) as {len(PRESETS) * len(ranges)} independent "
                                   f"(preset, block-range) tasks on {cores} threads"},
        "e2e": {"value": round(value, 4), "unit": "MSamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "detail": {str(m): {"enc_s": round(v[0], 4), "dec_s": round(v[1], 4), "bytes": v[2], "lossless": v[3]}
                   for m, v in sorted(last.items())},
    }
    print(json.dumps(line), flush=True)



# =================================================================================================
# at-scale legs (BASELINE.json configs[2] "C3" and the sharded-stream step of configs[4] "C5")
# =================================================================================================
def long_pcm(seconds):
    clip = make_clip()
    n = int(round(seconds * RATE))
    reps = (n + clip.shape[1] - 1) // clip.shape[1]
    return np.ascontiguousarray(np.tile(clip, (1, reps))[:, :n])


def cut_stream(stream, max_blocks):
    """header + the first `max_blocks` blocks of a stream, sample count patched (blocks are self-contained)."""
    off, ns, k = 30, 0, 0
    while off < len(stream) and k < max_blocks:
        size = int.from_bytes(stream[off + 2:off + 6], "big") + 6
        ns += int.from_bytes(stream[off + 9:off + 11], "big")
        off += size; k += 1
    hdr = bytearray(stream[:30]); hdr[14:18] = ns.to_bytes(4, "big")
    return bytes(hdr) + bytes(stream[30:off]), ns


def run_c3(args, dev, hbm_peak, fp64_peak):
    """C3: decode-only throughput on a synthetic 1-hour 44.1 kHz 16-bit stereo stream at -m 7 (the stream is
    built with the GPU encoder, whose m7 throughput is reported beside it)."""
    import torch
    import harness
    from linne_b200 import EncoderSession, DecoderSession
    pcm = long_pcm(args.c3_seconds)
    nch, n = pcm.shape
    stride = (n + 4 + 3) // 4 * 4
    h_pcm = torch.from_numpy(pcm).pin_memory()
    d_pcm = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    d_pcm[:, :n].copy_(h_pcm)
    cap = 30 + nch * n * 2 + 11 * (n // BLOCK + 2) + 65536
    d_stream = torch.zeros(cap + 64, dtype=torch.uint8, device=dev)
    enc = EncoderSession(nch, bits=BITS, rate=RATE, block=BLOCK, preset=7)
    dec = DecoderSession(channels=nch)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed_once(fn):
        torch.cuda.synchronize()
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    size = [0]
    def do_encode():
        size[0] = enc.encode_whole_resident(d_pcm.data_ptr(), stride, n, d_stream.data_ptr(), cap)
    do_encode()                                                  # warm-up: allocations
    enc.set_profiling(True); enc.reset_stage_stats()
    ms_enc = timed_once(do_encode)
    enc_stages = {k: round(v[1], 3) for k, v in sorted(enc.stage_stats().items(), key=lambda kv: -kv[1][1])}
    enc.set_profiling(False)
    sz = size[0]
    h_stream = torch.zeros(sz + 16, dtype=torch.uint8).pin_memory()
    h_stream[:sz].copy_(d_stream[:sz])
    d_back = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    h_back = torch.zeros((nch, n), dtype=torch.int32).pin_memory()
    chan_out = (C.POINTER(C.c_int32) * nch)(*[C.cast(h_back[c].data_ptr(), C.POINTER(C.c_int32)) for c in range(nch)])

    def dec_resident():          # stream and PCM stay in HBM; the host keeps a copy of the image for the block hop
        dec.decode_whole_resident(h_stream.data_ptr(), d_stream.data_ptr(), sz, d_back.data_ptr(), stride, nch, n)
    def dec_e2e():               # the reference call: host stream in, host PCM out
        dec.decode_whole(h_stream.data_ptr(), sz, chan_out, nch, n)
    dec_resident(); dec_e2e()                                    # warm-up
    dec.set_profiling(True); dec.reset_stage_stats()
    ms_res = min(timed_once(dec_resident) for _ in range(3))
    stages = dec.stage_stats()
    dec.set_profiling(False)
    ms_e2e = min(timed_once(dec_e2e) for _ in range(2))
    # packed-PCM call (SURVEY 8f.2): host stream in, interleaved 16-bit PCM out -- half the device->host bytes
    h_packed = torch.zeros(n * nch * (BITS // 8), dtype=torch.uint8).pin_memory()
    frames = C.c_uint32(0)
    u8p = C.POINTER(C.c_uint8)
    def dec_packed():
        rc = dec.lib.LINNEB200_DecodeWholePacked(dec.h, C.cast(h_stream.data_ptr(), u8p), sz, C.cast(h_packed.data_ptr(), u8p),
                                                 n, C.byref(frames))
        if rc != 0:
            raise RuntimeError(f"DecodeWholePacked rc={rc}")
    dec_packed()
    ms_packed = min(timed_once(dec_packed) for _ in range(2))
    ok_packed = bool(np.array_equal(h_packed.numpy().view("<i2").reshape(n, nch).T, pcm))
    ok = bool(torch.equal(d_back[:, :n], d_pcm[:, :n])) and bool(np.array_equal(h_back.numpy(), pcm)) and ok_packed
    samples = nch * n
    bytes_per_sample = 4.0 + sz / samples
    dec_stage_ms = {k: round(v[1] / 3.0, 3) for k, v in sorted(stages.items(), key=lambda kv: -kv[1][1])}
    dom = max(dec_stage_ms.items(), key=lambda kv: kv[1])
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            c3_traffic = json.load(f)
    except Exception:
        c3_traffic = {}
    out = {
        "workload": f"C3: {args.c3_seconds:.0f} s 44.1 kHz 16-bit stereo, -m 7, {n // BLOCK + 1} blocks, decode-only",
        "value": round(samples / (ms_res / 1e3) / 1e6, 1), "unit": "MSamples/s", "ms": round(ms_res, 3),
        "e2e": {"value": round(samples / (ms_e2e / 1e3) / 1e6, 1), "ms": round(ms_e2e, 3),
                "h2d_bytes": int(sz), "d2h_bytes": int(4 * samples)},
        "e2e_packed": {"value": round(samples / (ms_packed / 1e3) / 1e6, 1), "ms": round(ms_packed, 3),
                       "h2d_bytes": int(sz), "d2h_bytes": int((BITS // 8) * samples),
                       "call": "LINNEB200_DecodeWholePacked: interleaved 16-bit PCM out, converted on the device"},
        "stream_bytes": int(sz), "lossless": ok, "stages_ms": dec_stage_ms,
        "roofline": {"bound": "hbm", "kernel": dom[0], "achieved": round(bytes_per_sample * samples / (dom[1] / 1e3) / 1e9, 1),
                     "peak": hbm_peak, "unit": "GB/s",
                     "frac": round(bytes_per_sample * samples / (dom[1] / 1e3) / 1e9 / hbm_peak, 4),
                     "bytes_per_sample": round(bytes_per_sample, 3), "traffic": c3_traffic.get(dom[0]),
                     "traffic_note": "ncu dram bytes per launch on a stream of this size (profiles/ncu_traffic.json, r1_tput_ncu_full.md): "
                                     "the residuals make one pass through HBM between the two throughput kernels"},
        "encode_m7": {"value": round(samples / (ms_enc / 1e3) / 1e6, 1), "unit": "MSamples/s", "ms": round(ms_enc, 2),
                      "stages_ms": enc_stages,
                      "fp64_frac": round(2.0 * MAC_PER_SAMPLE[7] * samples / (enc_stages.get("analyze_v3", ms_enc) / 1e3) / 1e12
                                         / fp64_peak, 4) if fp64_peak else None},
    }
    # the reference decoder on the first blocks of the same stream, one host core
    try:
        if harness.have_ref():
            sub, ns = cut_stream(h_stream[:sz].numpy().tobytes(), 1024)
            ref = harness.Ref()
            t0 = time.perf_counter(); back = ref.decode(sub); dt = time.perf_counter() - t0
            out["cpu_baseline"] = {"value": round(nch * ns / dt / 1e6, 3), "unit": "MSamples/s", "cores": 1, "kind": "reference",
                                   "sample": f"reference decoder on the first 1024 blocks ({ns} frames), {dt:.1f} s",
                                   "matches": bool(np.array_equal(back, pcm[:, :ns]))}
    except Exception as e:  # pragma: no cover
        out["cpu_baseline"] = {"value": None, "kind": "unavailable", "sample": str(e)}
    enc.close(); dec.close()
    del d_pcm, d_stream, d_back, h_pcm, h_back, h_stream, h_packed
    torch.cuda.empty_cache()
    return out


def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2] if xs else None


def run_streaming(args, pcm):
    """SURVEY 8(f).4: the block-at-a-time callers (tools/linne_codec encodes with EncodeBlock per block,
    tools/linne_player decodes with DecodeBlock per block).  Host wall clock around every synchronous call, host buffers;
    DecodeBlock with and without read-ahead; the unmodified reference through the same calls beside it."""
    import torch
    import harness
    from harness import LINNEEncodeParameter, LINNEEncoderConfig, LINNEDecoderConfig
    from linne_b200 import Product
    nch, n = pcm.shape
    u8p, i32p = C.POINTER(C.c_uint8), C.POINTER(C.c_int32)
    impls = [("b200", Product())]
    if harness.have_ref():
        impls.append(("reference", harness.Ref()))
    out = {"workload": f"C2 clip block by block ({(n + BLOCK - 1) // BLOCK} blocks of {BLOCK} frames x {nch} ch), host buffers, "
                       "wall clock per synchronous call", "unit": "us per call (median)"}
    h_pcm = torch.from_numpy(pcm.copy()).pin_memory()
    cap = 2 * nch * BLOCK * 4 + 4096
    h_blk = torch.zeros(cap, dtype=torch.uint8).pin_memory()
    h_back = torch.zeros((nch, BLOCK), dtype=torch.int32).pin_memory()
    back_ptrs = (i32p * nch)(*[C.cast(h_back[c].data_ptr(), i32p) for c in range(nch)])
    for m in (0, 7):
        res = {}
        stream = None
        for name, impl in impls:
            L = impl.lib
            enc = L.LINNEEncoder_Create(C.byref(LINNEEncoderConfig(nch, BLOCK, 3, 128)), None, 0)
            L.LINNEEncoder_SetEncodeParameter(enc, C.byref(LINNEEncodeParameter(nch, BITS, RATE, BLOCK, m, 1, 0, 0)))
            size = C.c_uint32(0)
            for attempt in range(2 if name == "b200" else 1):                    # first pass warms the handle up
                lat, parts = [], []
                for lo in range(0, n, BLOCK):
                    k = min(BLOCK, n - lo)
                    ptrs = (i32p * nch)(*[C.cast(h_pcm[c].data_ptr() + 4 * lo, i32p) for c in range(nch)])
                    t0 = time.perf_counter()
                    rc = L.LINNEEncoder_EncodeBlock(enc, ptrs, k, C.cast(h_blk.data_ptr(), u8p), cap, C.byref(size))
                    lat.append(time.perf_counter() - t0)
                    if rc != 0:
                        raise RuntimeError(f"EncodeBlock rc={rc}")
                    parts.append(h_blk[:size.value].numpy().tobytes())
            L.LINNEEncoder_Destroy(enc)
            body = b"".join(parts)
            res[name + "_encode_block"] = round(1e6 * _median(lat), 1)
            res[name + "_encode_msamples_s"] = round(nch * n / sum(lat) / 1e6, 3)
            if name == "b200":
                stream = body
            h_img = torch.zeros(len(stream) + 16, dtype=torch.uint8).pin_memory()
            h_img[:len(stream)] = torch.frombuffer(bytearray(stream), dtype=torch.uint8)
            hdr = harness.LINNEHeader(1, 2, nch, n, RATE, BITS, BLOCK, m, 1)
            for k_ahead in ((0, 16) if name == "b200" else (0,)):
                dec = L.LINNEDecoder_Create(C.byref(LINNEDecoderConfig(nch, 3, 128, 1)), None, 0)
                L.LINNEDecoder_SetHeader(dec, C.byref(hdr))
                if name == "b200":
                    L.LINNEB200_DecoderSetReadahead(dec, k_ahead)
                used, got = C.c_uint32(0), C.c_uint32(0)
                for attempt in range(2 if name == "b200" else 1):
                    lat, off, done, ok = [], 0, 0, True
                    while off < len(stream):
                        t0 = time.perf_counter()
                        rc = L.LINNEDecoder_DecodeBlock(dec, C.cast(h_img.data_ptr() + off, u8p), len(stream) - off, back_ptrs, nch, BLOCK,
                                                        C.byref(used), C.byref(got))
                        lat.append(time.perf_counter() - t0)
                        if rc != 0:
                            raise RuntimeError(f"DecodeBlock rc={rc}")
                        ok = ok and bool(np.array_equal(h_back.numpy()[:, :got.value], pcm[:, done:done + got.value]))
                        off += used.value; done += got.value
                L.LINNEDecoder_Destroy(dec)
                tag = name + "_decode_block" + (f"_readahead{k_ahead}" if k_ahead else "")
                res[tag] = round(1e6 * _median(lat), 1)
                res[tag + "_mean"] = round(1e6 * sum(lat) / len(lat), 1)
                res[tag.replace("_block", "") + "_msamples_s"] = round(nch * n / sum(lat) / 1e6, 3)
                res[tag + "_lossless"] = ok and done == n
        out[f"m{m}"] = res
    return out


def run_c4(args, dev, fp64_peak):
    """C4 (BASELINE.json configs[3]): 24-bit 96 kHz 8-channel synthetic audio, encode at -m 7."""
    import torch
    import harness
    from linne_b200 import EncoderSession, DecoderSession, Product
    bits, rate, nch = 24, 96000, 8
    base = harness.synth_pcm(seconds=5.0, sr=rate, channels=nch, bits=bits, seed=4)
    reps = max(1, int(round(args.c4_seconds / 5.0)))
    pcm = np.ascontiguousarray(np.tile(base, (1, reps)))
    n = pcm.shape[1]
    stride = (n + 4 + 3) // 4 * 4
    samples = nch * n
    h_pcm = torch.from_numpy(pcm).pin_memory()
    d_pcm = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    d_pcm[:, :n].copy_(h_pcm)
    cap = 30 + nch * n * 3 + 11 * (n // BLOCK + 2) + 65536
    d_stream = torch.zeros(cap + 64, dtype=torch.uint8, device=dev)
    h_stream = torch.zeros(cap + 64, dtype=torch.uint8).pin_memory()
    enc = EncoderSession(nch, bits=bits, rate=rate, block=BLOCK, preset=7)
    dec = DecoderSession(channels=nch)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed_once(fn):
        torch.cuda.synchronize()
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    size = [0]
    chan_in = (C.POINTER(C.c_int32) * nch)(*[C.cast(h_pcm[c].data_ptr(), C.POINTER(C.c_int32)) for c in range(nch)])
    def enc_resident():
        size[0] = enc.encode_whole_resident(d_pcm.data_ptr(), stride, n, d_stream.data_ptr(), cap)
    def enc_e2e():
        size[0] = enc.encode_whole(chan_in, n, h_stream.data_ptr(), cap)
    enc_resident(); enc_e2e()
    enc.set_profiling(True); enc.reset_stage_stats()
    ms_res = min(timed_once(enc_resident) for _ in range(2))
    stages = {k: round(v[1] / 2.0, 3) for k, v in sorted(enc.stage_stats().items(), key=lambda kv: -kv[1][1])}
    enc.set_profiling(False)
    ms_e2e = min(timed_once(enc_e2e) for _ in range(2))
    sz = size[0]
    # packed 24-bit interleaved in (3 B per sample over PCIe instead of 4)
    packed = np.ascontiguousarray(pcm.T).astype("<i4").view(np.uint8).reshape(n, nch, 4)[:, :, :3]
    h_packed = torch.from_numpy(np.ascontiguousarray(packed).reshape(-1)).pin_memory()
    u8p = C.POINTER(C.c_uint8)
    osz = C.c_uint32(0)
    def enc_packed():
        rc = enc.lib.LINNEB200_EncodeWholePacked(enc.h, C.cast(h_packed.data_ptr(), u8p), n, C.cast(h_stream.data_ptr(), u8p), cap, C.byref(osz))
        if rc != 0:
            raise RuntimeError(f"EncodeWholePacked rc={rc}")
    enc_packed()
    ms_packed = min(timed_once(enc_packed) for _ in range(2))
    same_packed = osz.value == sz
    d_back = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    def dec_resident():
        dec.decode_whole_resident(None, d_stream.data_ptr(), sz, d_back.data_ptr(), stride, nch, n)
    enc_resident(); dec_resident()
    ms_dec = min(timed_once(dec_resident) for _ in range(2))
    ok = bool(torch.equal(d_back[:, :n], d_pcm[:, :n]))
    out = {
        "workload": f"C4: {n / rate:.0f} s 96 kHz 24-bit 8-channel synthetic, -m 7, {(n + BLOCK - 1) // BLOCK} blocks, encode",
        "value": round(samples / (ms_res / 1e3) / 1e6, 1), "unit": "MSamples/s", "ms": round(ms_res, 3),
        "e2e": {"value": round(samples / (ms_e2e / 1e3) / 1e6, 1), "ms": round(ms_e2e, 3), "h2d_bytes": int(4 * samples), "d2h_bytes": int(sz)},
        "e2e_packed": {"value": round(samples / (ms_packed / 1e3) / 1e6, 1), "ms": round(ms_packed, 3), "h2d_bytes": int(3 * samples),
                       "d2h_bytes": int(sz), "same_bytes": bool(same_packed)},
        "stream_bytes": int(sz), "ratio": round(sz / (3.0 * samples), 4), "lossless": ok, "stages_ms": stages,
        "fp64_frac": round(2.0 * MAC_PER_SAMPLE[7] * samples / (stages.get("analyze_v3", ms_res) / 1e3) / 1e12 / fp64_peak, 4) if fp64_peak else None,
        "decode": {"value": round(samples / (ms_dec / 1e3) / 1e6, 1), "ms": round(ms_dec, 3)},
    }
    try:
        if harness.have_ref():
            sub = np.ascontiguousarray(pcm[:, :2 * BLOCK])
            ref = harness.Ref()
            t0 = time.perf_counter(); rs = ref.encode(sub, bits=bits, rate=rate, preset=7); dt = time.perf_counter() - t0
            ours = Product().encode(sub, bits=bits, rate=rate, preset=7)
            out["cpu_baseline"] = {"value": round(sub.size / dt / 1e6, 4), "unit": "MSamples/s", "cores": 1, "kind": "reference",
                                   "sample": f"reference encoder -m 7 on the first 2 blocks x 8 ch ({sub.size} samples), {dt:.1f} s",
                                   "reference_bytes": len(rs), "b200_bytes": len(ours), "identical": bool(rs == ours)}
    except Exception as e:  # pragma: no cover
        out["cpu_baseline"] = {"value": None, "kind": "unavailable", "sample": repr(e)}
    enc.close(); dec.close()
    del d_pcm, d_stream, d_back, h_pcm, h_stream, h_packed
    torch.cuda.empty_cache()
    return out


def run_c5(args, dev, rank, world):
    """C5 (BASELINE.json configs[4]): a corpus of --c5-files stereo 16-bit 44.1 kHz files of 6 minutes each (1000 files =
    100 hours), sharded over the ranks by contiguous file (= block) ranges, encode AND decode of every file.
    No exchange between ranks.  The PCM of a few distinct files stays resident in HBM and is cycled (127 GB of int32
    PCM is not materialised); every file is a full EncodeWhole + DecodeWhole.  Time = max over ranks (CUDA events)."""
    import torch
    import torch.distributed as dist
    from linne_b200 import EncoderSession, DecoderSession
    clip = make_clip()
    nch = clip.shape[0]
    n = int(round(args.c5_file_seconds * RATE))
    reps = (n + clip.shape[1] - 1) // clip.shape[1]
    stride = (n + 4 + 3) // 4 * 4
    variants = []
    for v in range(3):
        x = np.ascontiguousarray(np.tile(np.roll(clip, 7919 * v, axis=1), (1, reps))[:, :n])
        d = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
        d[:, :n].copy_(torch.from_numpy(x))
        variants.append(d)
    samples_per_file = nch * n
    cap = 30 + nch * n * 2 + 11 * (n // BLOCK + 2) + 65536
    from linne_b200 import shard
    lo, hi = shard.file_ranges(args.c5_files, world)[rank]
    J = max(1, args.c5_workers)
    K = max(1, args.c5_batch)
    from linne_b200 import FileDesc
    if K > 1:
        d_corpus = torch.zeros((nch, K * stride), dtype=torch.int32, device=dev)      # K files side by side, variants cycled
        for s_ in range(K):
            d_corpus[:, s_ * stride:s_ * stride + stride].copy_(variants[s_ % len(variants)])
    out = {"workload": f"C5: {args.c5_files} files x {args.c5_file_seconds:.0f} s stereo 16-bit 44.1 kHz "
                       f"({args.c5_files * args.c5_file_seconds / 3600.0:.1f} h), {(n + BLOCK - 1) // BLOCK} blocks per file, "
                       "encode + decode of every file, files sharded by contiguous range over the ranks",
           "unit": "MSamples/s", "scaling": "strong", "workers_per_rank": J, "files_per_rank": hi - lo,
           "decoder_throughput_blocks": args.c5_tput_blocks, "files_per_call": K,
           "note": "samples counted once per file (a file that went through encode and decode counts once)"}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    for m, frac in ((0, 1.0), (7, args.c5_m7_fraction)):
        nfiles = max(J, int(round((hi - lo) * frac))) if frac > 0 else 0
        if nfiles == 0:
            continue
        total_files = nfiles * world if frac < 1.0 else args.c5_files
        encs = [EncoderSession(nch, bits=BITS, rate=RATE, block=BLOCK, preset=m) for _ in range(J)]
        decs = [DecoderSession(channels=nch) for _ in range(J)]
        for s_ in decs:                                             # several handles in flight: see include/linne_b200.h
            s_.lib.LINNEB200_DecoderSetThroughputBlocks(s_.h, args.c5_tput_blocks)
        last = [None] * J
        sizes = [0] * J
        errs = []
        if K > 1:
            # corpus batches: K files per call (LINNEB200_EncodeFilesResident / DecodeFilesResident)
            d_streams = [torch.zeros(K * cap + 64, dtype=torch.uint8, device=dev) for _ in range(J)]
            d_backs = [torch.zeros((nch, K * stride), dtype=torch.int32, device=dev) for _ in range(J)]
            descs = [(FileDesc * K)() for _ in range(J)]

            def work(j, count):
                try:
                    total = C.c_uint32(0)
                    lib = encs[j].lib
                    for b0 in range(j * K, count, J * K):
                        k = min(K, count - b0)
                        for s_ in range(k):
                            descs[j][s_] = FileDesc(s_ * stride, n, 0, 0, 0)
                        rc = lib.LINNEB200_EncodeFilesResident(encs[j].h, C.c_void_p(d_corpus.data_ptr()), K * stride, descs[j], k,
                                                               C.c_void_p(d_streams[j].data_ptr()), K * cap, C.byref(total))
                        rc = rc or lib.LINNEB200_DecodeFilesResident(decs[j].h, C.c_void_p(d_streams[j].data_ptr()), total.value, descs[j], k,
                                                                     C.c_void_p(d_backs[j].data_ptr()), K * stride)
                        if rc != 0:
                            raise RuntimeError(f"corpus batch rc={rc}")
                        last[j], sizes[j] = k, int(descs[j][0].out_size)
                except Exception as e:  # pragma: no cover
                    errs.append(e)

            def check(j):
                return last[j] is not None and all(bool(torch.equal(d_backs[j][:, s_ * stride:s_ * stride + n], d_corpus[:, s_ * stride:s_ * stride + n]))
                                                   for s_ in range(last[j]))
        else:
            d_streams = [torch.zeros(cap + 64, dtype=torch.uint8, device=dev) for _ in range(J)]
            d_backs = [torch.zeros((nch, stride), dtype=torch.int32, device=dev) for _ in range(J)]

            def work(j, count):
                try:
                    for f in range(j, count, J):
                        v = (lo + f) % len(variants)
                        sz = encs[j].encode_whole_resident(variants[v].data_ptr(), stride, n, d_streams[j].data_ptr(), cap)
                        decs[j].decode_whole_resident(None, d_streams[j].data_ptr(), sz, d_backs[j].data_ptr(), stride, nch, n)
                        last[j], sizes[j] = v, sz
                except Exception as e:  # pragma: no cover
                    errs.append(e)

            def check(j):
                return last[j] is not None and bool(torch.equal(d_backs[j][:, :n], variants[last[j]][:, :n]))

        def run(count):
            ts = [threading.Thread(target=work, args=(j, count)) for j in range(J)]
            for t in ts: t.start()
            for t in ts: t.join()
            if errs:
                raise errs[0]
        run(J * K)                                                  # warm-up: allocations
        barrier()
        e0.record(); run(nfiles); e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1))
        ok = all(check(j) for j in range(J))
        launches = sum(s.launch_count() for s in encs + decs)
        if m == 0:
            size_m0 = int(sizes[0])
        out[f"m{m}"] = {"files": total_files, "hours_of_audio": round(total_files * args.c5_file_seconds / 3600.0, 2),
                        "value": round(total_files * samples_per_file / (ms / 1e3) / 1e6, 1), "seconds": round(ms / 1e3, 3),
                        "ms_per_file_per_rank": round(ms / nfiles, 3), "lossless": ok, "bytes_last_file": int(sizes[0]),
                        "ratio": round(sizes[0] / (2.0 * samples_per_file), 4), "gpu_launches_rank0": int(launches)}
        for s in encs + decs:
            s.close()
        del d_streams, d_backs

    # ---- the file pipeline end to end (SURVEY 8f.3): packed PCM in host memory -> .lnn -> packed PCM in host memory ----
    # what linne_b200_cli does per file between its disk read and its disk write, with 1 and with 3 workers per rank
    if args.c5_e2e_files > 0:
        u8p = C.POINTER(C.c_uint8)
        host_pcm = torch.from_numpy(np.ascontiguousarray(variants[0][:, :n].cpu().numpy().T).astype("<i2").view(np.uint8).reshape(-1)).pin_memory()
        e2e = {}
        K2max = max(1, min(K, 4))
        host_pcm_k = host_pcm
        if K2max > 1:
            host_pcm_k = torch.zeros(K2max * host_pcm.numel(), dtype=torch.uint8).pin_memory()
            for s_ in range(K2max):
                host_pcm_k[s_ * host_pcm.numel():(s_ + 1) * host_pcm.numel()].copy_(host_pcm)
        for J2, K2 in ((1, 1), (3, 1), (3, K2max)):
            encs = [EncoderSession(nch, bits=BITS, rate=RATE, block=BLOCK, preset=0) for _ in range(J2)]
            decs = [DecoderSession(channels=nch) for _ in range(J2)]
            for s_ in decs:
                s_.lib.LINNEB200_DecoderSetThroughputBlocks(s_.h, args.c5_tput_blocks if J2 > 1 else 2560)
            h_lnn = [torch.zeros(K2 * cap, dtype=torch.uint8).pin_memory() for _ in range(J2)]
            h_out = [torch.zeros(K2 * host_pcm.numel(), dtype=torch.uint8).pin_memory() for _ in range(J2)]
            errs = []

            def work2(j, count):
                try:
                    sz, fr = C.c_uint32(0), C.c_uint32(0)
                    if K2 > 1:                                  # K2 files per call: LINNEB200_EncodeFilesPacked / DecodeFilesPacked
                        desc = (FileDesc * K2)()
                        for b0 in range(j * K2, count, J2 * K2):
                            k = min(K2, count - b0)
                            for s_ in range(k):
                                desc[s_] = FileDesc(0, n, 0, 0, 0)
                            rc = encs[j].lib.LINNEB200_EncodeFilesPacked(encs[j].h, C.cast(host_pcm_k.data_ptr(), u8p), desc, k,
                                                                         C.cast(h_lnn[j].data_ptr(), u8p), K2 * cap, C.byref(sz))
                            rc = rc or decs[j].lib.LINNEB200_DecodeFilesPacked(decs[j].h, C.cast(h_lnn[j].data_ptr(), u8p), sz.value, desc, k,
                                                                               C.cast(h_out[j].data_ptr(), u8p))
                            if rc != 0:
                                raise RuntimeError(f"packed corpus batch rc={rc}")
                        return
                    for f in range(j, count, J2):
                        rc = encs[j].lib.LINNEB200_EncodeWholePacked(encs[j].h, C.cast(host_pcm.data_ptr(), u8p), n,
                                                                     C.cast(h_lnn[j].data_ptr(), u8p), cap, C.byref(sz))
                        rc = rc or decs[j].lib.LINNEB200_DecodeWholePacked(decs[j].h, C.cast(h_lnn[j].data_ptr(), u8p), sz.value,
                                                                           C.cast(h_out[j].data_ptr(), u8p), n, C.byref(fr))
                        if rc != 0:
                            raise RuntimeError(f"packed call rc={rc}")
                except Exception as e:  # pragma: no cover
                    errs.append(e)

            def run2(count):
                ts = [threading.Thread(target=work2, args=(j, count)) for j in range(J2)]
                for t in ts: t.start()
                for t in ts: t.join()
                if errs:
                    raise errs[0]
            nf = max(J2 * K2, (args.c5_e2e_files // (J2 * K2)) * J2 * K2)      # whole batches for every worker
            run2(J2 * K2)
            barrier()
            e0.record(); run2(nf); e1.record()
            barrier()
            ms = max_over_ranks(e0.elapsed_time(e1))
            ok = all(bool(torch.equal(h[:host_pcm.numel()], host_pcm)) and bool(torch.equal(h[-host_pcm.numel():], host_pcm)) for h in h_out)
            tag = f"workers{J2}" + (f"_files_per_call{K2}" if K2 > 1 else "")
            e2e[tag] = {"value": round(world * nf * samples_per_file / (ms / 1e3) / 1e6, 1),
                        "ms_per_file_per_rank": round(ms / nf, 3), "files_per_rank": nf, "lossless": ok}
            for s in encs + decs:
                s.close()
            del h_lnn, h_out
        e2e["files_per_rank"] = args.c5_e2e_files
        e2e["preset"] = 0
        e2e["h2d_bytes_per_file"] = int(host_pcm.numel()) + size_m0
        e2e["d2h_bytes_per_file"] = int(host_pcm.numel()) + size_m0
        e2e["call"] = ("LINNEB200_EncodeWholePacked + LINNEB200_DecodeWholePacked on page-locked host buffers (what linne_b200_cli -j N runs "
                       "per file); files_per_call: LINNEB200_EncodeFilesPacked + LINNEB200_DecodeFilesPacked")
        out["e2e_pipeline_m0"] = e2e
    del variants
    torch.cuda.empty_cache()
    return out


def run_sharded(args, dev, rank, world):
    """One long stream sharded by contiguous block ranges over the ranks (SURVEY 8e), PCM ranges resident in HBM:
    every rank encodes its range at -m 7; shard byte counts are all-gathered and scanned; every rank writes its shard
    into rank 0's device buffer with one device-to-device copy through a CUDA IPC peer mapping (NVLink, no collective);
    then every rank decodes its own block range (no exchange).  Time = max over ranks, CUDA events."""
    import torch
    import torch.distributed as dist
    from linne_b200 import Product, shard, EncoderSession, DecoderSession, DeviceBuffer, PeerMapping
    pcm = long_pcm(args.shard_seconds)
    nch, n = pcm.shape
    lo, hi = shard.block_ranges(n, BLOCK, world)[rank]
    count = hi - lo
    stride = (count + 4 + 3) // 4 * 4
    d_pcm = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    d_pcm[:, :count].copy_(torch.from_numpy(np.ascontiguousarray(pcm[:, lo:hi])))
    cap = 30 + nch * count * 2 + 11 * (count // BLOCK + 2) + 65536
    d_shard = torch.zeros(cap + 64, dtype=torch.uint8, device=dev)
    d_back = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    enc = EncoderSession(nch, bits=BITS, rate=RATE, block=BLOCK, preset=7)
    dec = DecoderSession(channels=nch)
    res, dest, peer = {}, None, None
    # control plane, once, outside the timed region: rank 0's destination buffer (sized for the worst case of every
    # shard), its IPC handle to every rank, the peer mapping opened and kept
    caps_t = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(caps_t, torch.tensor([cap], dtype=torch.int64, device=dev))
    handle_t = torch.zeros(64, dtype=torch.uint8, device=dev)
    if rank == 0:
        dest = DeviceBuffer(30 + sum(int(t.item()) for t in caps_t) + 64)
        handle_t.copy_(torch.frombuffer(bytearray(dest.ipc_handle()), dtype=torch.uint8))
    dist.broadcast(handle_t, src=0)
    if rank != 0:
        peer = PeerMapping(bytes(handle_t.cpu().numpy().tobytes()))
    sizes_all = torch.zeros(world, dtype=torch.int64, device=dev)
    mine = torch.zeros(1, dtype=torch.int64, device=dev)
    for it in range(3):                                          # first passes warm allocations and the NVLink path
        torch.cuda.synchronize(); dist.barrier()
        e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        e0.record()
        size = enc.encode_whole_resident(d_pcm.data_ptr(), stride, count, d_shard.data_ptr(), cap) - 30
        mine.fill_(size)
        dist.all_gather_into_tensor(sizes_all, mine)             # 8 bytes per rank: the shard byte counts
        sizes = sizes_all.tolist()
        offsets, total = shard.exclusive_scan(sizes)
        if rank == 0:
            dest.lib.LINNEB200_DeviceCopy(dest.ptr + 30 + offsets[0], d_shard.data_ptr() + 30, size)
        else:
            peer.put(30 + offsets[rank], d_shard.data_ptr() + 30, size)
        torch.cuda.synchronize(); dist.barrier()
        e1.record()
        e2.record()
        dec.decode_whole_resident(None, d_shard.data_ptr(), size + 30, d_back.data_ptr(), stride, nch, count)
        e3.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1), e2.elapsed_time(e3)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ok = torch.tensor([1 if torch.equal(d_back[:, :count], d_pcm[:, :count]) else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        whole_ok = None
        if rank == 0:                                            # the gathered stream is ONE valid .lnn file
            hdr = shard.patch_num_samples(bytes(d_shard[:30].cpu().numpy().tobytes()), n)
            dest.upload(hdr, 0)
            if it == 2:
                whole = dest.download(30 + total)
                whole_ok = bool(np.array_equal(Product().decode(whole), pcm))
        res = {"workload": f"{args.shard_seconds:.0f} s stereo stream ({nch * n} samples), -m 7, contiguous block ranges over {world} GPUs, "
                           f"PCM ranges resident in HBM",
               "encode_gather_ms": round(float(t[0]), 2), "decode_ms": round(float(t[1]), 2),
               "encode_MSamples_s": round(nch * n / (float(t[0]) / 1e3) / 1e6, 1),
               "decode_MSamples_s": round(nch * n / (float(t[1]) / 1e3) / 1e6, 1),
               "stream_bytes": 30 + total, "lossless": bool(int(ok.item())), "gathered_stream_decodes": whole_ok,
               "exchange": "timed: all-gather of shard byte counts (8 B per rank) + exclusive scan + one device-to-device put per rank into "
                           "rank 0's buffer through a CUDA-IPC peer mapping opened once (NVLink); no data-path collective; "
                           "decode: every rank its own block range, no exchange"}
    enc.close(); dec.close()
    if peer is not None:
        peer.close()
    dist.barrier()
    if dest is not None:
        dest.free()
    return res


# =================================================================================================
# our arm
# =================================================================================================
def run_inlib_multi(args, dev):
    """Several GPUs behind ONE handle of ONE process (include/linne_b200.h: LINNEB200_*SetDevices; SURVEY 8e): the reference
    API's EncodeWhole / DecodeWhole on host buffers, a 600 s stereo stream at -m 7, on one device without and with
    pipelined block ranges and on every visible device.  Wall clock of the synchronous calls (median of 3)."""
    import torch
    import harness
    from linne_b200 import EncoderSession, DecoderSession
    pcm = long_pcm(args.shard_seconds)
    nch, n = pcm.shape
    cap = 30 + nch * n * 2 + 11 * (n // BLOCK + 2) + 65536
    h_pcm = torch.from_numpy(pcm.copy()).pin_memory()
    h_out = torch.zeros(cap, dtype=torch.uint8).pin_memory()
    h_back = torch.zeros((nch, n), dtype=torch.int32).pin_memory()
    chan_in = (C.POINTER(C.c_int32) * nch)(*[C.cast(h_pcm[c].data_ptr(), C.POINTER(C.c_int32)) for c in range(nch)])
    chan_out = (C.POINTER(C.c_int32) * nch)(*[C.cast(h_back[c].data_ptr(), C.POINTER(C.c_int32)) for c in range(nch)])
    visible = torch.cuda.device_count()
    out = {"workload": f"{args.shard_seconds:.0f} s stereo stream ({nch * n} samples), -m 7, host buffers through LINNEEncoder_EncodeWhole / "
                       f"LINNEDecoder_DecodeWhole, one process", "visible_gpus": visible, "unit": "ms per call (median of 3)"}
    reference_stream = None
    configs = [("one_device_no_pipeline", 1, "1"), ("one_device_pipelined", 1, None)]
    for g in (2, 4, 8):
        if g <= visible:
            configs.append((f"{g}_devices", g, None))
    for name, devices, pipeline in configs:
        if pipeline is None:
            os.environ.pop("LINNE_B200_PIPELINE", None)
        else:
            os.environ["LINNE_B200_PIPELINE"] = pipeline
        enc = EncoderSession(nch, bits=BITS, rate=RATE, block=BLOCK, preset=7)
        dec = DecoderSession(channels=nch)
        enc.set_devices(devices); dec.set_devices(devices)
        te, td = [], []
        for it in range(4):
            t0 = time.perf_counter(); size = enc.encode_whole(chan_in, n, h_out.data_ptr(), cap); t1 = time.perf_counter()
            h_back.zero_()
            t2 = time.perf_counter(); dec.decode_whole(h_out.data_ptr(), size, chan_out, nch, n); t3 = time.perf_counter()
            if it:
                te.append((t1 - t0) * 1e3); td.append((t3 - t2) * 1e3)
        stream = bytes(h_out[:size].numpy().tobytes())
        if reference_stream is None:
            reference_stream = stream
        out[name] = {"encode_ms": round(sorted(te)[1], 2), "decode_ms": round(sorted(td)[1], 2),
                     "encode_MSamples_s": round(nch * n / sorted(te)[1] / 1e3, 1), "decode_MSamples_s": round(nch * n / sorted(td)[1] / 1e3, 1),
                     "same_bytes_as_one_device": stream == reference_stream, "lossless": bool(np.array_equal(h_back.numpy(), pcm))}
        enc.close(); dec.close()
    os.environ.pop("LINNE_B200_PIPELINE", None)
    return out


def run_refine(args, dev, pcm, fp64_peak):
    """The non-default analysis paths (SURVEY rows a14, a15): IRLS (-a 3) and momentum SGD (-l) on the C2 clip at -m 0,
    device-resident; the refinement kernel's time against the FP64 pipe, the reference on a bounded sample beside it.
    FLOP counts: IRLS per iteration and unit n * p^2 / 2 (upper triangle of the weighted Gram matrix, lpc.c:452-509) +
    n * p (residual); SGD per iteration 3 * n * sum(P) (linne_network.c:805-873), 2 flops per multiply-add."""
    import torch
    import harness
    from linne_b200 import EncoderSession
    nch, n = pcm.shape
    stride = (n + 4 + 3) // 4 * 4
    cap = 30 + 2 * nch * n * 4 + 65536
    d_pcm = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    d_pcm[:, :n].copy_(torch.from_numpy(pcm.copy()))
    d_out = torch.zeros(cap + 64, dtype=torch.uint8, device=dev)
    out = {"workload": "C2 clip, -m 0, device-resident encode with the optional analysis paths", "unit": "MSamples/s"}
    layers = [2, 32]
    for name, opts in (("irls_a3", {"af": 3}), ("sgd_l", {"learning": 1})):
        enc = EncoderSession(nch, bits=BITS, rate=RATE, block=BLOCK, preset=0, **opts)
        enc.encode_whole_resident(d_pcm.data_ptr(), stride, n, d_out.data_ptr(), cap)           # warm-up
        enc.set_profiling(True); enc.reset_stage_stats()
        reps = 3
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            size = enc.encode_whole_resident(d_pcm.data_ptr(), stride, n, d_out.data_ptr(), cap)
        ms = (time.perf_counter() - t0) * 1e3 / reps
        st = enc.stage_stats()
        enc.close()
        k_ms = st.get("refine_v2", (1, 0.0))[1] / reps
        leg = {"value": round(nch * n / ms / 1e3, 2), "ms": round(ms, 3), "bytes": int(size), "refine_v2_ms": round(k_ms, 3),
               "stages_ms": {k: round(v[1] / reps, 3) for k, v in sorted(st.items(), key=lambda kv: -kv[1][1])}}
        if name == "irls_a3":
            # upper bound: every unit count 1, all 3 iterations run
            flops = 2.0 * nch * n * sum(3 * (P * P / 2.0 + 2 * P) for P in layers)
            leg["fp64_frac_upper"] = round(flops / (k_ms / 1e3) / 1e12 / fp64_peak, 5) if k_ms and fp64_peak else None
        try:
            impl = harness.Ref() if harness.have_ref() else harness.Oracle()
            sub = pcm[:, :4 * BLOCK]
            t0 = time.perf_counter()
            ref = impl.encode(sub, preset=0, **opts)
            dt = time.perf_counter() - t0
            from linne_b200 import Product
            mine = Product().encode(sub, preset=0, **opts)
            leg["reference"] = {"value": round(sub.size / dt / 1e6, 4), "cores": 1, "sample": f"first {sub.shape[1]} frames, {dt:.1f} s",
                                "bytes": len(ref), "b200_bytes": len(mine), "delta_pct": round(100.0 * (len(mine) - len(ref)) / len(ref), 4)}
        except Exception as e:  # pragma: no cover
            leg["reference"] = {"error": repr(e)}
        out[name] = leg
    return out


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import harness
    from linne_b200 import EncoderSession, DecoderSession, Product

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- linne_b200 has no CPU fallback")
    # Eight host threads per rank wait on their streams; when the ranks of a box outnumber its cores, spinning waits
    # starve each other, so the library's waits poll and yield the core between polls (LINNE_B200_SYNC=yield; measured on a
    # 32-core box: 4 GPUs 4.45 ms per sweep against 5.0 ms with sleeping waits and 4.55 ms spinning, 8 GPUs 4.89 against
    # 5.25 ms -- profiles/RESULTS.md).
    oversubscribed = world * len(PRESETS) > 0.75 * (os.cpu_count() or 1)
    sync_mode_forced = oversubscribed and "LINNE_B200_SYNC" not in os.environ
    if oversubscribed:
        os.environ.setdefault("LINNE_B200_SYNC", args.oversub_wait)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"            # keep NCCL's version banner off stdout (one JSON line)
        dist.init_process_group("nccl", device_id=dev)
    product = Product()
    hbm_peak, peak_src = load_peaks()

    pcm = make_clip()
    nch, n = pcm.shape
    n_samples = nch * n
    stride = (n + 4 + 3) // 4 * 4
    cap = 30 + 2 * nch * n * 4 + 65536

    # host (pinned) and device buffers
    h_pcm = torch.from_numpy(pcm.copy()).pin_memory()
    d_pcm = torch.zeros((nch, stride), dtype=torch.int32, device=dev)
    d_pcm[:, :n].copy_(h_pcm)
    d_out = [torch.zeros(cap + 64, dtype=torch.uint8, device=dev) for _ in PRESETS]
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    # one encoder + one decoder handle per preset, each with its own CUDA stream: the sweep's eight
    # presets are independent streams of work, so a server would run them side by side
    encs = {m: EncoderSession(nch, bits=BITS, rate=RATE, block=BLOCK, preset=m) for m in PRESETS}
    decs = {m: DecoderSession(channels=nch) for m in PRESETS}
    h_outs = {m: torch.zeros(cap, dtype=torch.uint8).pin_memory() for m in PRESETS}
    h_backs = {m: torch.zeros((nch, n), dtype=torch.int32).pin_memory() for m in PRESETS}
    d_backs = {m: torch.zeros((nch, stride), dtype=torch.int32, device=dev) for m in PRESETS}
    chan_outs = {m: (C.POINTER(C.c_int32) * nch)(*[C.cast(h_backs[m][c].data_ptr(), C.POINTER(C.c_int32)) for c in range(nch)])
                 for m in PRESETS}

    chan_in = (C.POINTER(C.c_int32) * nch)(*[C.cast(h_pcm[c].data_ptr(), C.POINTER(C.c_int32)) for c in range(nch)])
    sizes = {}

    # --schedule phased: the eight presets encode side by side, meet, then decode side by side.  The analysis kernel takes
    # a whole SM per CTA (224 KB of shared memory) while a decode CTA lives ~0.8 ms on a quarter of one: interleaved, the
    # early presets' decode CTAs spread over the SMs and keep the late presets' analysis CTAs waiting for an empty SM.
    phase_gate = threading.Barrier(len(PRESETS)) if (args.schedule == "phased" and not args.serial and args.sweep_threads >= len(PRESETS)) else None

    def one_e2e(m):
        sz = encs[m].encode_whole(chan_in, n, h_outs[m].data_ptr(), cap)
        sizes[m] = sz
        if phase_gate is not None and not args.serial:
            phase_gate.wait()
        decs[m].decode_whole(h_outs[m].data_ptr(), sz, chan_outs[m], nch, n)

    def one_resident(m):
        sz = encs[m].encode_whole_resident(d_pcm.data_ptr(), stride, n, d_out[m].data_ptr(), cap)
        sizes[m] = sz
        if phase_gate is not None and not args.serial:
            phase_gate.wait()
        # host image = None: the decoder fetches the (1 MB) stream image itself to hop over the block
        # size fields -- inside the timed region
        decs[m].decode_whole_resident(None, d_out[m].data_ptr(), sz, d_backs[m].data_ptr(), stride, nch, n)

    # The sweep's host threads live as long as the bench (a server's workers): a step releases them and meets them again,
    # so thread creation (~0.1 ms each under the interpreter lock) is not part of a step.
    class SweepPool:
        def __init__(self):
            self.fn = None; self.errs = []; self.stop = False
            # --sweep-threads T < 8: thread j runs presets 7 - j, then j, ... (a cheap one after an expensive one)
            T = max(1, min(len(PRESETS), args.sweep_threads))
            order = PRESETS[::-1]                                  # longest presets first
            self.lists = [[] for _ in range(T)]
            for i, m in enumerate(order):
                j = i % (2 * T)
                self.lists[j if j < T else 2 * T - 1 - j].append(m)
            self.go = threading.Barrier(T + 1); self.done = threading.Barrier(T + 1)
            self.threads = [threading.Thread(target=self.work, args=(ms,), daemon=True) for ms in self.lists]
            for t in self.threads: t.start()

        def work(self, ms):
            while True:
                self.go.wait()
                if self.stop:
                    return
                try:
                    for m in ms:
                        self.fn(m)
                except Exception as e:      # pragma: no cover
                    self.errs.append(e)
                    if phase_gate is not None:
                        phase_gate.abort()
                self.done.wait()

        def run(self, fn):
            self.fn = fn
            self.go.wait(); self.done.wait()
            if self.errs:
                raise self.errs[0]

        def close(self):
            self.stop = True
            self.go.wait()
            for t in self.threads: t.join(timeout=2)
    pool = SweepPool()

    def run_sweep(one):
        if args.serial:
            for m in PRESETS:
                one(m)
            return
        pool.run(one)

    def step_e2e():
        run_sweep(one_e2e)

    def step_resident():
        run_sweep(one_resident)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, profile=False):
        for _ in range(warmup):
            fn()
        if profile:
            for s in list(encs.values()) + list(decs.values()):
                s.set_profiling(True); s.reset_stage_stats()
        launches0 = sum(s.launch_count() for s in list(encs.values()) + list(decs.values()))
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(steps):
            l2_flush.fill_(1)                       # flush L2 between timed iterations
            torch.cuda.current_stream().synchronize()
            fn()                                    # every API call is synchronous: all its device work is done on return
        t1.record()
        barrier()
        ms = t0.elapsed_time(t1) / steps
        launches = sum(s.launch_count() for s in list(encs.values()) + list(decs.values())) - launches0
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, launches // steps

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_res, launches = timed(step_resident, args.steps, args.warmup, profile=True)
    sampler.stop_flag.set(); sampler.join(timeout=3)
    if args.dump_outputs and rank == 0:         # before the legs below run the same handles again
        dump_outputs(args.dump_outputs, {m: d_out[m][:sizes[m]] for m in PRESETS}, {m: d_backs[m][:, :n] for m in PRESETS})

    # correctness of what was just timed (outside the timed region)
    torch.cuda.synchronize()
    ok_resident = all(bool(torch.equal(d_backs[m][:, :n].cpu(), h_pcm)) for m in PRESETS)
    stage = {}
    for sess in list(encs.values()) + list(decs.values()):
        for name, (cnt, ms) in sess.stage_stats().items():
            a = stage.setdefault(name, [0, 0.0]); a[0] += cnt; a[1] += ms
        sess.set_profiling(False)

    ms_e2e, _ = timed(step_e2e, args.steps, args.warmup)
    ok_e2e = all(bool(np.array_equal(h_backs[m].numpy(), pcm)) for m in PRESETS)
    comp_bytes = dict(sizes)

    value = len(PRESETS) * n_samples * world / (ms_res / 1e3) / 1e6
    e2e_value = len(PRESETS) * n_samples * world / (ms_e2e / 1e3) / 1e6
    h2d = sum(4 * n_samples + comp_bytes[m] for m in PRESETS)     # PCM up for encode, stream up for decode
    d2h = sum(comp_bytes[m] + 4 * n_samples for m in PRESETS)     # stream down from encode, PCM down from decode

    # ---- roofline of the dominant kernel ----
    # Per-kernel durations come from CUDA events recorded on each launching stream.  In the timed region the
    # eight presets overlap, so a kernel's event time there includes the other streams' kernels it shared the
    # GPU with; the roofline therefore uses a SERIAL pass of the same step (same inputs, profiling on, kernels
    # alone on the GPU) run right after the timed region.  Both sets of stage times are reported.
    args_serial = args.serial
    args.serial = True
    for sess in list(encs.values()) + list(decs.values()):
        sess.set_profiling(True); sess.reset_stage_stats()
    serial_steps = max(1, min(args.steps, 3))
    torch.cuda.synchronize()
    for _ in range(serial_steps):
        l2_flush.fill_(1); torch.cuda.current_stream().synchronize()
        step_resident()
    stage_serial = {}
    for sess in list(encs.values()) + list(decs.values()):
        for name, (cnt, ms) in sess.stage_stats().items():
            a = stage_serial.setdefault(name, [0, 0.0]); a[0] += cnt; a[1] += ms
        sess.set_profiling(False)
    args.serial = args_serial

    fp64_peak = product.measure_fp64_tflops() if rank == 0 else 0.0
    total_comp = sum(comp_bytes.values())
    hbm_bytes_per_sample = 4.0 + total_comp / (len(PRESETS) * n_samples)      # SURVEY 8(d): int32 PCM + compressed bytes
    analysis_kernels = {"analyze_v3", "to_double", "acorr", "solve", "loss", "select", "forward", "refine_v2"}
    dec_kernels = {"crc_v2", "stream_v2", "tp_entropy", "tp_synth", "entropy_v3", "synth_v2", "crc", "entropy", "synth", "deemph", "ms_inverse"}
    dom = max(stage_serial.items(), key=lambda kv: kv[1][1]) if stage_serial else ("none", [1, 1.0])
    dom_name, (dom_cnt, dom_ms) = dom[0], dom[1]
    try:        # DRAM bytes per launch of that kernel from the committed ncu capture (profiles/)
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            traffic = json.load(f).get(dom_name)
    except Exception:
        traffic = None
    samples_done = len(PRESETS) * n_samples * serial_steps
    if dom_name in analysis_kernels:
        flops = 2.0 * sum(MAC_PER_SAMPLE[m] for m in PRESETS) * n_samples * serial_steps
        achieved = flops / (dom_ms / 1e3) / 1e12
        roofline = {"bound": "fp64", "kernel": dom_name, "achieved": round(achieved, 4), "peak": round(fp64_peak, 3),
                    "unit": "TFLOP/s", "frac": round(achieved / fp64_peak, 5) if fp64_peak else None, "traffic": traffic,
                    "traffic_source": "static: profiles/ncu_traffic.json (ncu --set full captures named there), not re-measured by this run",
                    "launches": dom_cnt, "avg_launch_ms": round(dom_ms / max(dom_cnt, 1), 4),
                    "note": "encoder analysis is FP64-pipe bound (SURVEY 8d): algorithmic FLOPs = 2 x MAC/sample table "
                            "(un-deduplicated) over this kernel's summed launch time; peak = DFMA microbenchmark on this GPU"}
    else:
        by = hbm_bytes_per_sample * samples_done
        achieved = by / (dom_ms / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom_name, "achieved": round(achieved, 3), "peak": hbm_peak,
                    "unit": "GB/s", "frac": round(achieved / hbm_peak, 5), "traffic": traffic, "peak_source": peak_src,
                    "traffic_source": "static: profiles/ncu_traffic.json (ncu --set full captures named there), not re-measured by this run",
                    "traffic_note": "ncu dram bytes per launch at -m 7 (profiles/ncu_traffic.json); algorithmic bytes per launch = "
                                    + str(int(hbm_bytes_per_sample * n_samples)),
                    "launches": dom_cnt, "avg_launch_ms": round(dom_ms / max(dom_cnt, 1), 4),
                    "bytes_per_sample": round(hbm_bytes_per_sample, 3),
                    "note": "latency-bound at this batch size (44 blocks per launch): serial by format, one pipeline of warps per block"}
    # the other side of the path, always reported: encoder analysis against the FP64 pipe, decode against HBM
    an_ms = sum(v[1] for k, v in stage_serial.items() if k in analysis_kernels)
    flops = 2.0 * sum(MAC_PER_SAMPLE[m] for m in PRESETS) * n_samples * serial_steps
    roofline_analysis = {"bound": "fp64", "kernels": sorted(k for k in stage_serial if k in analysis_kernels),
                         "achieved": round(flops / (an_ms / 1e3) / 1e12, 4) if an_ms else None, "peak": round(fp64_peak, 3),
                         "unit": "TFLOP/s", "frac": round(flops / (an_ms / 1e3) / 1e12 / fp64_peak, 5) if an_ms and fp64_peak else None}
    dec_ms = sum(v[1] for k, v in stage_serial.items() if k in dec_kernels)
    by = hbm_bytes_per_sample * samples_done
    roofline_decode = {"bound": "hbm", "kernels": sorted(k for k in stage_serial if k in dec_kernels),
                       "achieved": round(by / (dec_ms / 1e3) / 1e9, 3) if dec_ms else None,
                       "peak": hbm_peak, "unit": "GB/s", "frac": round(by / (dec_ms / 1e3) / 1e9 / hbm_peak, 5) if dec_ms else None,
                       "peak_source": peak_src, "bytes_per_sample": round(hbm_bytes_per_sample, 3)}

    # ---- per mode and per direction (BASELINE.json's metric is quoted per -m mode): every preset alone on the GPU,
    #      wall clock of the synchronous calls (median), device-resident and through host buffers ----
    per_mode = {}
    pm_reps = max(3, min(args.steps, 7))

    def _median_ms(fn):
        ts = []
        for _ in range(pm_reps):
            l2_flush.fill_(1); torch.cuda.synchronize()
            t0 = time.perf_counter(); fn(); ts.append((time.perf_counter() - t0) * 1e3)
        return sorted(ts)[len(ts) // 2]
    for m in PRESETS:
        sz = sizes[m]
        enc_res = _median_ms(lambda: encs[m].encode_whole_resident(d_pcm.data_ptr(), stride, n, d_out[m].data_ptr(), cap))
        dec_res = _median_ms(lambda: decs[m].decode_whole_resident(None, d_out[m].data_ptr(), sz, d_backs[m].data_ptr(), stride, nch, n))
        enc_h = _median_ms(lambda: encs[m].encode_whole(chan_in, n, h_outs[m].data_ptr(), cap))
        dec_h = _median_ms(lambda: decs[m].decode_whole(h_outs[m].data_ptr(), sz, chan_outs[m], nch, n))
        per_mode[str(m)] = {"enc_MSps": round(n_samples / enc_res / 1e3, 1), "dec_MSps": round(n_samples / dec_res / 1e3, 1),
                            "enc_e2e_MSps": round(n_samples / enc_h / 1e3, 1), "dec_e2e_MSps": round(n_samples / dec_h / 1e3, 1),
                            "enc_ms": round(enc_res, 3), "dec_ms": round(dec_res, 3), "bytes": int(sz)}

    # ---- at-scale legs: free the sweep's buffers first ----
    host_wait_sweep = os.environ.get("LINNE_B200_SYNC", "spin")
    pool.close()
    for sess in list(encs.values()) + list(decs.values()):
        sess.close()
    if sync_mode_forced:
        del os.environ["LINNE_B200_SYNC"]                # the legs below choose for their own thread counts
    user_sync_mode = "LINNE_B200_SYNC" in os.environ

    def choose_host_wait(threads_per_rank):
        """sleeping waits only when the waiting host threads of the box outnumber its cores: a sleeping wait costs a
        wake-up per synchronisation, which the short per-file call chains of these legs feel"""
        if user_sync_mode:
            return os.environ["LINNE_B200_SYNC"]
        if world * threads_per_rank > (os.cpu_count() or 1):
            os.environ["LINNE_B200_SYNC"] = args.oversub_wait
            return args.oversub_wait
        os.environ.pop("LINNE_B200_SYNC", None)
        return "spin"
    del d_out, d_backs, h_outs, h_backs, l2_flush
    torch.cuda.empty_cache()
    sharded = None
    if world > 1 and args.shard_seconds > 0:
        try:
            choose_host_wait(1)
            sharded = run_sharded(args, dev, rank, world)
        except Exception as e:      # pragma: no cover
            sharded = {"error": repr(e)}
    c5 = None
    if args.c5_files > 0:
        try:
            wait_mode = choose_host_wait(max(1, args.c5_workers))      # read by the handles when they are created
            c5 = run_c5(args, dev, rank, world)
            c5["host_wait"] = wait_mode
        except Exception as e:      # pragma: no cover
            c5 = {"error": repr(e)}
        choose_host_wait(1)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    c4 = streaming = None
    if world == 1 and args.c4_seconds > 0:
        try:
            c4 = run_c4(args, dev, fp64_peak)
        except Exception as e:      # pragma: no cover
            c4 = {"error": repr(e)}
    if world == 1 and not args.no_streaming:
        try:
            streaming = run_streaming(args, pcm)
        except Exception as e:      # pragma: no cover
            streaming = {"error": repr(e)}
    inlib = None
    if world == 1 and args.shard_seconds > 0 and not args.no_inlib:
        try:
            inlib = run_inlib_multi(args, dev)
        except Exception as e:      # pragma: no cover
            inlib = {"error": repr(e)}
    refine = None
    if world == 1 and not args.no_refine:
        try:
            refine = run_refine(args, dev, pcm, fp64_peak)
        except Exception as e:      # pragma: no cover
            refine = {"error": repr(e)}
    c3 = None
    if world == 1 and args.c3_seconds > 0:
        try:
            c3 = run_c3(args, dev, hbm_peak, fp64_peak)
        except Exception as e:      # pragma: no cover
            c3 = {"error": repr(e)}

    # ---- CPU baseline beside it: the unmodified reference, one thread, bounded sample ----
    cpu_baseline = None
    try:
        impl, kind = (harness.Ref(), "reference") if harness.have_ref() else (harness.Oracle(), "port")
        sample_presets = [0, 4, 7]
        sub = pcm[:, :5 * BLOCK * 4]           # 20 full blocks = 4.64 s of the clip
        t0 = time.perf_counter()
        ref_sizes = {}
        for m in sample_presets:
            s = impl.encode(sub, preset=m); impl.decode(s); ref_sizes[m] = len(s)
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": round(len(sample_presets) * sub.size / dt / 1e6, 4), "unit": "MSamples/s", "cores": 1,
                        "kind": kind, "sample": f"first {sub.shape[1]} frames of the clip, presets {sample_presets}, "
                                                f"encode+decode, {dt:.1f} s of CPU work"}
    except Exception as e:  # pragma: no cover
        cpu_baseline = {"value": None, "unit": "MSamples/s", "cores": 1, "kind": "unavailable", "sample": str(e)}

    # ---- the reference's compressed size of the whole clip at every mode (one host thread per mode), beside ours ----
    try:
        impl_sz = harness.Ref if harness.have_ref() else harness.Oracle
        full_ref = {}

        def _ref_size(m):
            full_ref[m] = len(impl_sz().encode(pcm, preset=m))
        ths = [threading.Thread(target=_ref_size, args=(m,)) for m in PRESETS[::-1]]
        for t in ths: t.start()
        for t in ths: t.join()
        for m in PRESETS:
            pm = per_mode[str(m)]
            pm["ref_bytes"] = int(full_ref[m])
            pm["delta_pct"] = round(100.0 * (pm["bytes"] - full_ref[m]) / full_ref[m], 5)
    except Exception as e:  # pragma: no cover
        per_mode["ref_bytes_error"] = repr(e)

    line = {
        "metric": "encode+decode MSamples/s over the -m 0..7 sweep", "value": round(value, 3), "unit": "MSamples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_res, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic",
        "config": {"workload": "C2: 10 s 44.1 kHz 16-bit stereo synthetic clip, -m 0..7 sweep, encode+decode",
                   "block": BLOCK, "ms": 1, "presets": PRESETS, "l2": "256 MiB flush write between timed iterations",
                   "per_rank": "each rank runs the whole sweep on its own clip",
                   "concurrency": "serial" if args.serial else f"8 presets on {max(1, min(8, args.sweep_threads))} persistent host threads / CUDA streams", "schedule": args.schedule,
                   "host_wait": host_wait_sweep, "host_cores": os.cpu_count()},
        "e2e": {"value": round(e2e_value, 3), "unit": "MSamples/s", "ms_per_step": round(ms_e2e, 3),
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": int(launches),
        "roofline": roofline, "roofline_analysis": roofline_analysis, "roofline_decode": roofline_decode,
        "cpu_baseline": cpu_baseline,
        "clocks": sampler.summary(),
        "stages_ms_per_step": {k: round(v[1] / args.steps, 3) for k, v in sorted(stage.items(), key=lambda kv: -kv[1][1])},
        "stages_ms_per_step_serial": {k: round(v[1] / serial_steps, 3) for k, v in sorted(stage_serial.items(), key=lambda kv: -kv[1][1])},
        "per_mode": per_mode,
        "compressed_bytes": {str(m): int(comp_bytes[m]) for m in PRESETS},
        "lossless": {"resident": ok_resident, "e2e": ok_e2e},
        "fp64_peak_tflops": round(fp64_peak, 3),
    }
    if c3 is not None:
        line["c3_decode"] = c3
    if sharded is not None:
        line["sharded_stream"] = sharded
    if c4 is not None:
        line["c4_encode"] = c4
    if c5 is not None:
        line["c5_corpus"] = c5
    if streaming is not None:
        line["streaming"] = streaming
    if refine is not None:
        line["refine"] = refine
    if inlib is not None:
        line["inlib_multi_gpu"] = inlib
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--serial", action="store_true", help="run the eight presets one after the other (one stream)")
    ap.add_argument("--schedule", default="interleaved", choices=["interleaved", "phased"],
                    help="order of the sweep's calls: every preset encodes then decodes on its own thread (interleaved), or all "
                         "presets encode, meet, and then all decode (phased)")
    ap.add_argument("--oversub-wait", default="yield", choices=["block", "yield", "spin"],
                    help="host wait mode (LINNE_B200_SYNC) chosen when the waiting threads of the box outnumber its cores")
    ap.add_argument("--sweep-threads", type=int, default=8, help="host threads (CUDA streams in flight) the sweep's eight presets run on")
    ap.add_argument("--sweep-only", action="store_true", help="skip every leg but the headline sweep")
    ap.add_argument("--with-inlib", action="store_true", help="with --sweep-only: keep the in-library multi-GPU / pipelining leg")
    ap.add_argument("--c3-seconds", type=float, default=3600.0,
                    help="N=1: length of the C3 decode-only stream (BASELINE.json configs[2]); 0 = skip")
    ap.add_argument("--shard-seconds", type=float, default=600.0,
                    help="N>1: length of the stream sharded by block range over the ranks; 0 = skip")
    ap.add_argument("--c4-seconds", type=float, default=60.0,
                    help="N=1: length of the C4 clip (24-bit 96 kHz 8 ch, -m 7 encode; BASELINE.json configs[3]); 0 = skip")
    ap.add_argument("--c5-files", type=int, default=1000,
                    help="files of the C5 corpus (BASELINE.json configs[4]), sharded over the ranks; 0 = skip")
    ap.add_argument("--c5-file-seconds", type=float, default=360.0)
    ap.add_argument("--c5-m7-fraction", type=float, default=0.1, help="share of each rank's files also run at -m 7 (bounded)")
    ap.add_argument("--c5-workers", type=int, default=4, help="handle pairs (host threads / CUDA streams) per rank in the C5 leg")
    ap.add_argument("--c5-batch", type=int, default=8,
                    help="C5 leg: files per call (LINNEB200_EncodeFilesResident / DecodeFilesResident); 1 = one call per file")
    ap.add_argument("--c5-tput-blocks", type=int, default=1024,
                    help="C5 leg: LINNEB200_DecoderSetThroughputBlocks of its decoders (several handles in flight)")
    ap.add_argument("--c5-e2e-files", type=int, default=24, help="files per rank of the host-buffer pipeline leg; 0 = skip")
    ap.add_argument("--no-streaming", action="store_true", help="skip the EncodeBlock / DecodeBlock latency leg")
    ap.add_argument("--no-refine", action="store_true", help="skip the IRLS / SGD leg")
    ap.add_argument("--no-inlib", action="store_true", help="skip the in-library multi-GPU / pipelining leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the compressed streams and (a fixed sample of) the decoded PCM of the last timed sweep step "
                         "to DIR/<name>.npy (float32, rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 sweep")
    if args.sweep_only:
        args.c3_seconds = args.c4_seconds = 0.0
        if not args.with_inlib:
            args.shard_seconds = 0.0
        args.c5_files = 0
        args.no_streaming = args.no_refine = True
        args.no_inlib = not args.with_inlib
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
