"""Streams written with caller-chosen block parameters, against every decoder path and the forced-parameter encoder.

An encoder's analysis only ever picks a narrow slice of what the format allows: unit counts that divide the taps and the
analysis length, small coefficients with short Huffman codes, residuals far below 2^31, partition orders and Rice
parameters that follow smooth signals.  Here the oracle's `lo_encode_block_forced` writes every block with chosen unit
counts, shifts, int8 taps and pre-emphasis coefficients instead, so the special cases of the decoders are driven on
purpose: p >= 8, 4, 2, 1 taps per unit and more units than taps, units shorter than their taps, samples behind the last
unit, the longest coefficient codes, Rice parameters 0 and 30 side by side, partition orders 0 and 10, and residual code
words longer than 64 and than 4096 bits.

Every case first checks itself: the oracle decodes it back to its input, no partition has k2 = 31 (where the reference
shifts by 32, DESIGN section 2), and the feature it was built for really occurs.  `test_feature_coverage` checks that the
cases together reach every feature listed in REQUIRED.
"""
import ctypes as C
import functools
import os
from dataclasses import dataclass, field

import numpy as np
import pytest

import harness
from linne_b200.api import PRESET_LAYERS, ChannelParams, _chan_ptrs

SHAPE_PRESETS = (0, 2, 7)               # one preset per layer shape: (2, 32), (4, 64, 8), (4, 128, 16)
TPUT_FORMS = ("i", "8", "w", "l", "s")  # LINNE_B200_TP_ENTROPY


# ----------------------------------------------------------------------------------------------
# The generator
# ----------------------------------------------------------------------------------------------
@dataclass
class ChannelBlock:
    """What one channel of one block was written with, and what the oracle's coder made of it."""
    nsmp: int
    log2_units: list
    rshift: list
    coef: list                  # per layer, the P taps
    preem_coef: tuple
    preem_prev: tuple
    residual: np.ndarray
    porder: int
    k2: list                    # one per partition
    longest_code: int           # bits of the longest residual code word


@dataclass
class Forced:
    stream: bytes
    blocks: list                # [block][channel] -> ChannelBlock
    oracle_types: list = field(default_factory=list)   # block types of the oracle's own analysis (preem="oracle")


def _zz(x):
    x = np.asarray(x, dtype=np.int64)
    return np.where(x < 0, -2 * x - 1, 2 * x)


def _longest_code(residual, porder, k2):
    """length of the longest Rice code word of the residual under the coder's plan (oracle coder_emit)"""
    uv = _zz(residual)
    k = np.repeat(np.asarray(k2, np.int64), len(residual) >> porder)
    short = uv < (np.int64(1) << (k + 1))
    lens = np.where(short, k + 2, k + 2 + ((uv - (np.int64(1) << (k + 1))) >> k))
    return int(lens.max())


@functools.lru_cache(maxsize=None)
def _oracle():
    o = harness.Oracle()
    o.lib.lo_encoder_last_block_type.restype = C.c_int
    o.lib.lo_encoder_last_residual.restype = C.POINTER(C.c_int32)
    return o


def forced_stream(pcm, bits, preset, block, params_of, preem="forced"):
    """One stream whose every block is one lo_encode_block_forced call.

    params_of(block_index, channel) -> (log2_units, rshift, taps, preem_coef): per layer of the preset the log2 of the
    unit count, the shift and the P int8 taps; preem_coef is a pair in 0..15.  With preem="oracle" the pair is ignored
    and the oracle's own pre-emphasis coefficients of an unforced encode of the same block are used (what the GPU
    encoder computes for itself), and the oracle's block types are recorded.  The header is that of the oracle's own
    encode of the same shape with num_samples patched."""
    o = _oracle()
    L = o.lib
    pcm = np.ascontiguousarray(pcm, dtype=np.int32)
    nch, n = pcm.shape
    layers = PRESET_LAYERS[preset]
    ms = 1 if nch >= 2 else 0
    hdr = bytearray(o.encode(pcm[:, :1], bits=bits, preset=preset, block=block)[:30])
    hdr[14:18] = n.to_bytes(4, "big")
    enc = L.lo_encoder_create(nch, block)
    cap = 64 + 2 * nch * block * 8
    buf = np.zeros(cap, np.uint8)
    u8 = buf.ctypes.data_as(C.POINTER(C.c_uint8))
    size = C.c_uint32(0)
    out, blocks, types = [bytes(hdr)], [], []
    try:
        assert L.lo_encoder_configure(enc, nch, bits, 44100, block, preset, ms, 0, 0) == harness.OK
        for b, b0 in enumerate(range(0, n, block)):
            sub = np.ascontiguousarray(pcm[:, b0:b0 + block])
            m = sub.shape[1]
            trs = (harness.LoChannelTrace * nch)()
            if preem == "oracle":
                assert L.lo_encode_block(enc, _chan_ptrs(sub), m, u8, cap, C.byref(size)) == harness.OK
                types.append(L.lo_encoder_last_block_type(enc))
                oracle_pc = [tuple(L.lo_encoder_trace(enc, c).contents.preem_coef) for c in range(nch)]
            for c in range(nch):
                lu, rs, taps, pc = params_of(b, c)
                if preem == "oracle":
                    pc = oracle_pc[c]
                for l, P in enumerate(layers):
                    trs[c].num_units[l] = 1 << lu[l]
                    trs[c].rshift[l] = rs[l]
                    assert len(taps[l]) == P
                    for i in range(P):
                        trs[c].coef[l][i] = int(taps[l][i])
                trs[c].preem_coef[0], trs[c].preem_coef[1] = pc
            assert L.lo_encode_block_forced(enc, _chan_ptrs(sub), m, trs, u8, cap, C.byref(size)) == harness.OK
            out.append(buf[:size.value].tobytes())
            chans = []
            for c in range(nch):
                tr = L.lo_encoder_trace(enc, c).contents
                res = np.ctypeslib.as_array(L.lo_encoder_last_residual(enc, c), shape=(m,)).copy()
                po = C.c_uint32(0)
                k2 = np.zeros(1024, np.uint32)
                L.lo_coder_plan(res.ctypes.data_as(C.POINTER(C.c_int32)), m, C.byref(po),
                                k2.ctypes.data_as(C.POINTER(C.c_uint32)))
                k2 = [int(v) for v in k2[:1 << po.value]]
                chans.append(ChannelBlock(
                    nsmp=m, log2_units=[(int(tr.num_units[l]) - 1).bit_length() for l in range(len(layers))],
                    rshift=[int(tr.rshift[l]) for l in range(len(layers))],
                    coef=[[int(tr.coef[l][i]) for i in range(P)] for l, P in enumerate(layers)],
                    preem_coef=(int(tr.preem_coef[0]), int(tr.preem_coef[1])),
                    preem_prev=(int(tr.preem_prev[0]), int(tr.preem_prev[1])),
                    residual=res, porder=int(po.value), k2=k2, longest_code=_longest_code(res, po.value, k2)))
            blocks.append(chans)
    finally:
        L.lo_encoder_destroy(enc)
    return Forced(b"".join(out), blocks, types)


def channel_params(forced):
    """The ChannelParams records (block-major) that make EncodeWholeWithParams write what the oracle wrote."""
    nch = len(forced.blocks[0])
    arr = (ChannelParams * (len(forced.blocks) * nch))()
    for b, chans in enumerate(forced.blocks):
        for c, cb in enumerate(chans):
            p = arr[b * nch + c]
            for l in range(len(cb.coef)):
                p.log2_units[l] = cb.log2_units[l]
                p.rshift[l] = cb.rshift[l]
                for i, t in enumerate(cb.coef[l]):
                    p.coef[l][i] = t
    return arr


# ----------------------------------------------------------------------------------------------
# Features
# ----------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def longest_code_taps():
    """int8 taps whose coefficient code is the longest of the table (14 bits)"""
    _, lens = _oracle().coef_table()
    taps = [t for t in range(-128, 128) if lens[(2 * t if t >= 0 else -2 * t - 1) & 0xFF] == lens.max()]
    assert lens.max() == 14 and taps
    return tuple(taps)


def features(case, forced):
    got = set()
    layers = PRESET_LAYERS[case.preset]
    for b, chans in enumerate(forced.blocks):
        for cb in chans:
            n = cb.nsmp
            for l, P in enumerate(layers):
                U = 1 << cb.log2_units[l]
                p, m = P // U, n // U
                got.add(("units", layers, l, cb.log2_units[l]))
                if U <= P and m <= p:
                    got.add("unit shorter than its taps")
                if U <= P and m > p and n % U:
                    got.add("samples behind the last unit")
                got.add(("rshift", cb.rshift[l]))
                got.update(("tap", t) for t in (-128, 127) if t in cb.coef[l])
                if all(t in longest_code_taps() for t in cb.coef[l]):
                    got.add("every tap a 14-bit code")
            got.add(("preem", cb.preem_coef))
            if any(_zz(v) >> case.bits for v in cb.preem_prev):
                got.add("preem_prev fills bits + 1")
            got.update(("k2", k) for k in (0, 30) if k in cb.k2)
            if len(cb.k2) > 1 and np.abs(np.diff(cb.k2)).max() >= 25:
                got.add("k2 jump >= 25")
            got.add(("porder", cb.porder))
            if cb.longest_code > 64 and n == 10240:
                got.add("code word > 64 bits in a full 10240-sample block")
            if cb.longest_code > 4096:
                got.add("code word > 4096 bits")
    return got


REQUIRED = ({("units", PRESET_LAYERS[s], l, lu) for s in SHAPE_PRESETS for l in range(len(PRESET_LAYERS[s]))
             for lu in range(8)}
            | {"unit shorter than its taps", "samples behind the last unit", ("rshift", 0), ("rshift", 15),
               ("tap", -128), ("tap", 127), "every tap a 14-bit code", ("preem", (0, 0)), ("preem", (15, 15)),
               "preem_prev fills bits + 1", ("k2", 0), ("k2", 30), "k2 jump >= 25", ("porder", 0), ("porder", 10),
               "code word > 64 bits in a full 10240-sample block", "code word > 4096 bits"})


# ----------------------------------------------------------------------------------------------
# The cases
# ----------------------------------------------------------------------------------------------
@dataclass
class Case:
    name: str
    bits: int
    preset: int
    block: int
    make: object                # make(seed) -> (pcm, params_of)
    expect: frozenset = frozenset()    # features this case is built for
    encoder: bool = True        # the oracle's own analysis codes every block compressed: usable for encoder parity
    reseed: bool = False        # wrapping residuals: retry seeds until no partition has k2 = 31

    @property
    def tput_eligible(self):
        """the throughput decoder takes this stream (tails still go to the fused kernel in the same call)"""
        return self.block % 1024 == 0 and self.block <= 10240


def _random_params(preset, seed, log2_units=None, rshifts=(0, 1, 7, 15), taps="int8", preem=None):
    layers = PRESET_LAYERS[preset]

    def params_of(b, c):
        r = np.random.default_rng([seed, b, c])
        lu = [log2_units(b, l) if log2_units else int(r.integers(0, 8)) for l in range(len(layers))]
        rs = [rshifts[(b + l + c) % len(rshifts)] for l in range(len(layers))]
        if taps == "int8":
            tp = [r.integers(-128, 128, P) for P in layers]
        elif taps == "small":
            tp = [r.integers(-3, 4, P) for P in layers]
        elif taps == "zero":
            tp = [np.zeros(P, int) for P in layers]
        else:                   # "extreme": -128/127 and the longest codes, a layer each, alternating per block
            long_taps = longest_code_taps()
            tp = [np.where(np.arange(P) % 2, 127, -128) if (b + l) % 2 else
                  np.array([long_taps[(i + b) % len(long_taps)] for i in range(P)]) for l, P in enumerate(layers)]
        pc = preem if preem is not None else (int(r.integers(0, 16)), int(r.integers(0, 16)))
        return lu, rs, tp, pc
    return params_of


def _units_sweep(preset, channels, bits):
    def make(seed):
        pcm = harness.synth_pcm(n=4096 * 8 + 4095, channels=channels, bits=bits, seed=100 + preset + seed)
        return pcm, _random_params(preset, seed, log2_units=lambda b, l: (b + l) % 8)
    return make


def _short_tail(preset, tail):
    def make(seed):
        pcm = harness.synth_pcm(n=1024 * 2 + tail, channels=2, bits=16, seed=200 + tail + seed)
        return pcm, _random_params(preset, seed, taps="small", rshifts=(2, 4, 0, 15))
    return make


def _extremes(preset, channels):
    def make(seed):
        pcm = harness.synth_pcm(n=4096 * 3 + 777, channels=channels, bits=24, seed=300 + preset + seed)
        pcm[0, ::4096] = -(1 << 23)                        # full-scale first samples: with M/S the side channel
        if channels > 1:                                  # needs all 25 bits of its preem_prev field
            pcm[1, ::4096] = (1 << 23) - 1
        return pcm, _random_params(preset, seed, taps="extreme", rshifts=(15, 0, 15), preem=(15, 15))
    return make


def _stretches(n, bits, period, seed):
    """alternating digital silence and full-scale noise, `period` samples each, silence first"""
    r = np.random.default_rng(seed)
    x = r.integers(-(1 << (bits - 1)), 1 << (bits - 1), n)
    x[(np.arange(n) // period) % 2 == 0] = 0
    return x


def _quiet_loud_porder10(seed):
    pcm = _stretches(10240 * 2, 16, 10, seed)[None, :].astype(np.int32)
    return pcm, _random_params(0, seed, taps="zero", preem=(0, 0))


def _quiet_loud_wrap(seed):
    x = _stretches(4096 * 2 + 1024, 24, 512, seed)
    pcm = np.stack([x, x // 3]).astype(np.int32)
    # 127 * (two noise samples) wraps: partitions of the loud stretches reach k2 = 30 beside k2 = 0 of the silent ones
    return pcm, lambda b, c: ([0, 0], [0, 0], [np.array([127, 127]), np.zeros(32, int)], (0, 0))


def _click(block, tail, bits, where):
    def make(seed):
        r = np.random.default_rng(seed)
        n = 2 * block + tail
        pcm = r.integers(-1, 2, size=(1, n)).astype(np.int32)
        full = (1 << (bits - 1)) - 1
        if where == "full":     # alone in its 10-sample partition: 73 bits for 16-bit input
            pcm[0, block + 333] = full
        else:                   # an odd-length tail has one partition: one k2 for all of it
            pcm[0, 2 * block + tail // 2:2 * block + tail // 2 + 2] = full, -full
        return pcm, _random_params(0, seed, log2_units=lambda b, l: 0, taps="zero", preem=(0, 0))
    return make


def _format(preset, channels, bits, block, tail):
    def make(seed):
        pcm = harness.synth_pcm(n=block * 3 + tail, channels=channels, bits=bits, seed=400 + channels + seed)
        return pcm, _random_params(preset, seed, taps="small", rshifts=(0, 3, 15, 1))
    return make


def _long_block(preset):
    def make(seed):
        pcm = harness.synth_pcm(n=16384 * 2 + 5000, channels=2, bits=16, seed=500 + preset + seed)
        return pcm, _random_params(preset, seed, log2_units=lambda b, l: (3 * b + l) % 8)
    return make


CASES = (
    [Case(f"units_sweep_m{p}_stereo16", 16, p, 4096, _units_sweep(p, 2, 16), reseed=True,
          expect=frozenset({("units", PRESET_LAYERS[p], l, lu) for l in range(len(PRESET_LAYERS[p])) for lu in range(8)}
                           | {("rshift", 0), ("rshift", 15), "samples behind the last unit"})) for p in SHAPE_PRESETS]
    + [Case(f"units_sweep_m{p}_mono24", 24, p, 4096, _units_sweep(p, 1, 24), reseed=True) for p in SHAPE_PRESETS]
    + [Case(f"short_tail_{t}_m{SHAPE_PRESETS[i % 3]}", 16, SHAPE_PRESETS[i % 3], 1024, _short_tail(SHAPE_PRESETS[i % 3], t),
            expect=frozenset({"unit shorter than its taps"}) if t < 32 else frozenset())
       for i, t in enumerate((1, 2, 7, 8, 9, 31, 33, 100, 127, 129))]
    + [Case(f"extremes_m{p}_stereo24", 24, p, 4096, _extremes(p, 2), reseed=True,
            expect=frozenset({("tap", -128), ("tap", 127), "every tap a 14-bit code", ("preem", (15, 15)),
                              "preem_prev fills bits + 1"})) for p in SHAPE_PRESETS]
    + [Case("extremes_m7_mono24", 24, 7, 4096, _extremes(7, 1), reseed=True)]
    + [Case("quiet_loud_porder10", 16, 0, 10240, _quiet_loud_porder10, encoder=False,
            expect=frozenset({("porder", 10), ("k2", 0), ("preem", (0, 0))})),
       Case("quiet_loud_wrapping_taps", 24, 0, 4096, _quiet_loud_wrap, encoder=False, reseed=True,
            expect=frozenset({("k2", 0), ("k2", 30), "k2 jump >= 25"})),
       Case("click_full_10240_16bit", 16, 0, 10240, _click(10240, 0, 16, "full"), encoder=False,
            expect=frozenset({"code word > 64 bits in a full 10240-sample block"})),
       Case("click_odd_tail_4095_16bit", 16, 0, 4096, _click(4096, 4095, 16, "tail"), encoder=False,
            expect=frozenset({"code word > 4096 bits", ("porder", 0)})),
       Case("click_odd_tail_10239_24bit", 24, 0, 10240, _click(10240, 10239, 24, "tail"), encoder=False,
            expect=frozenset({"code word > 4096 bits"}))]
    + [Case("format_mono8_m7", 8, 7, 2048, _format(7, 1, 8, 2048, 1001)),
       Case("format_3ch24_ms_m2", 24, 2, 4096, _format(2, 3, 24, 4096, 1500)),
       Case("format_8ch16_m0", 16, 0, 1024, _format(0, 8, 16, 1024, 333))]
    + [Case(f"long_block_16384_m{p}", 16, p, 16384, _long_block(p), reseed=True) for p in (0, 7)])
CASE_BY_NAME = {c.name: c for c in CASES}
NAMES = [c.name for c in CASES]
ENCODER_NAMES = [c.name for c in CASES if c.encoder]


@functools.lru_cache(maxsize=None)
def built(name, preem="forced"):
    """(case, pcm, Forced) of a case; a case with wrapping residuals takes the first seed without a k2 = 31 partition"""
    case = CASE_BY_NAME[name]
    for seed in range(20 if case.reseed else 1):
        pcm, params_of = case.make(seed)
        forced = forced_stream(pcm, case.bits, case.preset, case.block, params_of, preem)
        if all(max(cb.k2) <= 30 for chans in forced.blocks for cb in chans):
            break
    return case, pcm, forced


def checked(name, preem="forced"):
    """built(), after the guard every comparison rests on"""
    case, pcm, forced = built(name, preem)
    rc, out = _oracle().decode(forced.stream, return_code=True)
    assert rc == harness.OK and np.array_equal(out, pcm), "the oracle does not decode the forced stream to its input"
    worst = max(max(cb.k2) for chans in forced.blocks for cb in chans)
    assert worst <= 30, "a partition has k2 = 31, where the reference's shift is undefined"
    if preem == "forced":
        missing = case.expect - features(case, forced)
        assert not missing, f"{name} does not reach what it was built for: {sorted(map(str, missing))}"
    else:
        # the GPU encoder decides the block type itself: the comparison means something only where it must say compressed
        assert forced.oracle_types == [0] * len(forced.blocks), forced.oracle_types
    return case, pcm, forced


@pytest.mark.parametrize("name", NAMES)
def test_forced_case_guard(name):
    checked(name)


def test_feature_coverage():
    reached = set()
    for case in CASES:
        reached |= features(case, built(case.name)[2])
    missing = sorted(map(str, REQUIRED - reached))
    assert not missing, f"no case reaches: {missing}"


# ----------------------------------------------------------------------------------------------
# Host simulator (the product's host code and kernel bodies on the CPU)
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_hostsim_decode_equals_oracle(hostsim, name):
    case, pcm, forced = checked(name)
    rc, out = hostsim.decode(forced.stream, return_code=True)
    assert rc == harness.OK
    assert np.array_equal(out, pcm)


@pytest.mark.parametrize("name", ENCODER_NAMES)
def test_hostsim_encode_with_params_equals_oracle(hostsim, name):
    case, pcm, forced = checked(name, preem="oracle")
    got = hostsim.encode_with_params(pcm, channel_params(forced), bits=case.bits, block=case.block, preset=case.preset)
    assert got == forced.stream


def _check_out_of_range_fields(codec, field_name, bad, top):
    """A field the stream cannot hold is rejected before anything is written; the largest one it holds is accepted."""
    case, pcm, forced = checked("units_sweep_m2_stereo16", preem="oracle")
    for value, accepted in ((bad, False), (top, True)):
        prm = channel_params(forced)
        getattr(prm[len(prm) - 1], field_name)[2] = value          # the last record, the preset's last layer
        rc, out = codec.encode_with_params(pcm, prm, bits=case.bits, block=case.block, preset=case.preset,
                                           return_code=True)
        if accepted:
            assert rc == harness.OK and np.array_equal(_oracle().decode(out), pcm), (field_name, value)
        else:
            assert (rc, out) == (harness.INVALID_ARGUMENT, b""), (field_name, value, rc)


OUT_OF_RANGE = [("log2_units", 8, 7), ("log2_units", 255, 7), ("rshift", 16, 15), ("rshift", 255, 15)]


@pytest.mark.parametrize("field_name,bad,top", OUT_OF_RANGE)
def test_hostsim_encode_with_params_rejects_fields_the_stream_cannot_hold(hostsim, field_name, bad, top):
    _check_out_of_range_fields(hostsim, field_name, bad, top)


# ----------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------
@pytest.fixture
def env_switch():
    """set environment switches the library reads per handle or per call, restored afterwards"""
    saved = {}

    def setenv(name, value):
        saved.setdefault(name, os.environ.get(name))
        os.environ[name] = value
    yield setenv
    for name, old in saved.items():
        if old is None:
            os.environ.pop(name, None)
        else:
            os.environ[name] = old


_LEG_DEFAULTS = {"LINNE_B200_TPUT_MIN_BLOCKS": "0", "LINNE_B200_WALK": "lane", "LINNE_B200_SPLIT_DECODE": "0",
                 "LINNE_B200_TP_ENTROPY": "i"}
# (leg, switches, stages that must run, stages that must not)
DECODE_LEGS = ([("fused", {}, {"stream_v2"}, {"tp_entropy"}),
                ("fused warp walk", {"LINNE_B200_WALK": "warp"}, {"stream_v2"}, {"tp_entropy"}),
                ("split", {"LINNE_B200_SPLIT_DECODE": "1"}, {"entropy_v3", "synth_v2"}, {"stream_v2", "tp_entropy"})]
               + [(f"throughput {f}", {"LINNE_B200_TPUT_MIN_BLOCKS": "1", "LINNE_B200_TP_ENTROPY": f},
                   {"tp_entropy", "tp_synth"}, set()) for f in TPUT_FORMS])


def _gpu_decode(stream, channels):
    """(result code, PCM, names of the stages that ran) of one DecodeWhole on a fresh handle"""
    from linne_b200 import DecoderSession
    dec = DecoderSession(channels=channels)
    try:
        dec.set_profiling(True)
        nch, n = int.from_bytes(stream[12:14], "big"), int.from_bytes(stream[14:18], "big")
        out = np.zeros((nch, n), np.int32)
        buf = np.frombuffer(stream, np.uint8)
        rc = dec.lib.LINNEDecoder_DecodeWhole(dec.h, buf.ctypes.data_as(C.POINTER(C.c_uint8)), len(stream),
                                              _chan_ptrs(out), nch, n)
        return rc, out, set(dec.stage_stats())
    finally:
        dec.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_gpu_decode_paths_equal_oracle(gpu, env_switch, name):
    case, pcm, forced = checked(name)
    tput = case.tput_eligible and not (pcm.shape[0] >= 2 and pcm.shape[0] % 2)     # M/S with odd C: not eligible
    legs = [leg for leg in DECODE_LEGS if tput or not leg[0].startswith("throughput")]
    for leg, switches, must, must_not in legs:
        for var, value in {**_LEG_DEFAULTS, **switches}.items():
            env_switch(var, value)
        rc, out, stages = _gpu_decode(forced.stream, pcm.shape[0])
        assert must <= stages and not (must_not & stages), (leg, sorted(stages))
        assert rc == harness.OK, (leg, rc)
        bad = np.nonzero((out != pcm).any(axis=0))[0]
        assert bad.size == 0, f"{leg}: {bad.size} frames differ, first at {bad[0]} (block {bad[0] // case.block})"


def _gpu_encode_with_params(case, pcm, params):
    """(result code, stream, names of the stages that ran) of one EncodeWholeWithParams"""
    from linne_b200 import EncoderSession
    nch, n = pcm.shape
    sess = EncoderSession(nch, bits=case.bits, block=case.block, preset=case.preset)
    try:
        sess.set_profiling(True)
        cap = 30 + 2 * nch * n * 4 + 4096
        out = np.zeros(cap, np.uint8)
        size = C.c_uint32(0)
        rc = sess.lib.LINNEB200_EncodeWholeWithParams(sess.h, _chan_ptrs(pcm), n, params, len(params) // nch,
                                                      out.ctypes.data_as(C.POINTER(C.c_uint8)), cap, C.byref(size))
        return rc, out[:size.value].tobytes(), set(sess.stage_stats())
    finally:
        sess.close()


def _block_spans(stream):
    spans, off = [], 30
    while off < len(stream):
        size = int.from_bytes(stream[off + 2:off + 6], "big") + 6
        spans.append(stream[off:off + size])
        off += size
    return spans


@pytest.mark.gpu
@pytest.mark.parametrize("name", ENCODER_NAMES)
def test_gpu_encode_with_params_equals_oracle(gpu, name):
    case, pcm, forced = checked(name, preem="oracle")
    rc, got, stages = _gpu_encode_with_params(case, pcm, channel_params(forced))
    # blocks of up to 10240 samples take the cooperative kernels, longer ones the flat items
    must = {"prepare_v2", "predict_plan_v2", "pack_v2"} if case.block <= 10240 else {"prepare", "predict", "plan"}
    assert must <= stages, sorted(stages)
    assert rc == harness.OK
    if got != forced.stream:
        gb, wb = _block_spans(got), _block_spans(forced.stream)
        differ = [i for i in range(max(len(gb), len(wb))) if gb[i:i + 1] != wb[i:i + 1]]
        units = [[cb.log2_units for cb in forced.blocks[i]] for i in differ[:4]]
        pytest.fail(f"blocks {differ} differ from the oracle's; log2_units of the first: {units}")


@pytest.mark.gpu
@pytest.mark.parametrize("field_name,bad,top", OUT_OF_RANGE)
def test_gpu_encode_with_params_rejects_fields_the_stream_cannot_hold(gpu, field_name, bad, top):
    _check_out_of_range_fields(gpu, field_name, bad, top)
