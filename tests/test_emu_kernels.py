"""CPU execution of the real CUDA kernel bodies (bzip3_b200/csrc/cm.cuh, lzp_parallel.cuh) on the
thread-block emulator of tests/native/cta_emu.h, compared bit-for-bit with the oracle.

This is the "no GPU in this container" safety net for the warp-/CTA-cooperative kernels: every CUDA thread
is a fiber, barriers and warp collectives are the switch points (see cta_emu.h for the limits: it proves
the protocol and the arithmetic, not the absence of races and nothing about speed).  The GPU parity tests
in test_gpu_parity.py remain the real gate."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from bzip3_b200 import synth
from tests import refs

ROOT = refs.ROOT
SO = os.path.join(ROOT, "tests", "_build", "libemucheck.so")
SRCS = [os.path.join(ROOT, "tests", "native", f) for f in ("emu_check.cpp", "cta_emu.cpp")]
DEPS = SRCS + [os.path.join(ROOT, "tests", "native", "cta_emu.h")] + [
    os.path.join(ROOT, "bzip3_b200", "csrc", f) for f in ("common.cuh", "cm.cuh", "lzp.cuh", "lzp_parallel.cuh")]

_lib = None


def emu():
    global _lib
    if _lib is None:
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        if not os.path.exists(SO) or any(os.path.getmtime(d) > os.path.getmtime(SO) for d in DEPS):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-x", "c++",
                                   "-o", SO] + SRCS)
        L = C.CDLL(SO)
        L.emu_set_schedule.argtypes = [C.c_int, C.c_ulonglong]
        L.emu_cm_encode.restype = C.c_int32
        L.emu_cm_encode.argtypes = [refs.u8p, C.c_int32, refs.u8p]
        L.emu_cm_decode.restype = C.c_int
        L.emu_cm_decode.argtypes = [refs.u8p, C.c_int32, refs.u8p, C.c_int32]
        L.emu_lzp_decode.restype = C.c_int32
        L.emu_lzp_decode.argtypes = [refs.u8p, C.c_int32, refs.u8p, C.c_int32, refs.i32p]
        _lib = L
    return _lib


def arr(b):
    return np.frombuffer(bytes(b), dtype=np.uint8).copy()


def bwt_of(data: np.ndarray) -> np.ndarray:
    """What the entropy stage really sees: the BWT of the data (oracle)."""
    O = refs.oracle()
    n = len(data)
    out = np.zeros(n + 16, np.uint8)
    O.orc_bwt(refs.ptr(data), refs.ptr(out), n)
    return out[:n].copy()


def cm_inputs():
    rng = np.random.default_rng(99)
    cases = [(name, arr(d)[:1200]) for name, d in synth.edge_cases() if len(d) > 0]
    cases.append(("bwt_zipf_12k", bwt_of(synth.zipf_text(12 << 10, seed=7))))
    cases.append(("bwt_source_10k", bwt_of(synth.source_corpus(10 << 10, seed=8))))
    cases.append(("random_6k", rng.integers(0, 256, 6000, dtype=np.uint8)))
    cases.append(("runs_8k", np.repeat(rng.integers(0, 4, 80, dtype=np.uint8), 100)))
    cases.append(("one_byte", np.array([65], np.uint8)))
    return cases


CM_CASES = cm_inputs()
CM_IDS = [c[0] for c in CM_CASES]


@pytest.mark.parametrize("name,data", CM_CASES, ids=CM_IDS)
def test_cm_encode_kernel(name, data):
    E, O = emu(), refs.oracle()
    n = len(data)
    want = np.zeros(2 * n + 64, np.uint8)
    got = np.zeros(2 * n + 64, np.uint8)
    rw = O.orc_cm_encode(refs.ptr(data), n, refs.ptr(want))
    rg = E.emu_cm_encode(refs.ptr(data), n, refs.ptr(got))
    assert rg == rw
    assert bytes(got[:rg]) == bytes(want[:rw])


@pytest.mark.parametrize("name,data", CM_CASES, ids=CM_IDS)
def test_cm_decode_kernel(name, data):
    E, O = emu(), refs.oracle()
    n = len(data)
    enc = np.zeros(2 * n + 64, np.uint8)
    r = O.orc_cm_encode(refs.ptr(data), n, refs.ptr(enc))
    # the whole stream, a truncated stream (read_in() past the end adds -1) and an empty one
    for insize in ((r, max(r - 3, 0), 0) if n <= 2000 else (r, r // 2)):
        want = np.zeros(n + 8, np.uint8)
        got = np.zeros(n + 8, np.uint8)
        O.orc_cm_decode(refs.ptr(enc), insize, refs.ptr(want), n)
        assert E.emu_cm_decode(refs.ptr(enc), insize, refs.ptr(got), n) == 0
        assert bytes(got[:n]) == bytes(want[:n]), (insize, r)
        if insize == r:
            assert bytes(got[:n]) == bytes(data)


def test_cm_decode_exhausted_streams():
    """Once the payload is exhausted read_in() feeds -1 (src/libbz3.c:345) and low <= code <= high no longer holds; the
    kernel's shortcuts (one renormalisation test per byte, range < 2^24 as the cheap pre-test) are switched off from
    there on, so truncated and garbage payloads decode exactly like the reference -- for as long as the caller asks."""
    E, O = emu(), refs.oracle()
    n, payloads = exhausted_payloads()
    pins = refs.reference_answer("cm_exhausted")   # the oracle itself is pinned on the reference for these payloads
    assert len(pins) == len(payloads)
    for (buf, insize), pin in zip(payloads, pins):
        want = np.zeros(n + 8, np.uint8)
        got = np.zeros(n + 8, np.uint8)
        O.orc_cm_decode(refs.ptr(buf), insize, refs.ptr(want), n)
        assert refs.digest(want[:n]) == pin, insize
        assert E.emu_cm_decode(refs.ptr(buf), insize, refs.ptr(got), n) == 0
        assert bytes(got[:n]) == bytes(want[:n]), insize


def exhausted_payloads():
    """(n, [(payload, insize)]): a CM payload cut short at many places, and garbage of a few bytes, decoded to n bytes."""
    O = refs.oracle()
    rng = np.random.default_rng(31337)
    data = CM_CASES[CM_IDS.index("bwt_zipf_12k")][1][:1500]
    n = len(data)
    enc = np.zeros(2 * n + 64, np.uint8)
    r = O.orc_cm_encode(refs.ptr(data), n, refs.ptr(enc))
    payloads = [(enc, cut) for cut in list(range(0, 12)) + [r // 7, r // 3, r - 9, r - 5, r - 4, r - 2, r - 1]]
    for k in range(24):   # garbage of a few bytes, decoded far past its end
        g = np.zeros(64, np.uint8)
        m = int(rng.integers(1, 40))
        g[:m] = rng.integers(0, 256, m, dtype=np.uint8) if k % 3 else np.full(m, 255 * (k % 2), np.uint8)
        payloads.append((g, m))
    return n, payloads


@pytest.mark.parametrize("schedule", [1, 2])
def test_cm_kernels_other_schedules(schedule):
    """Same result when the fibers are scheduled in descending or pseudo-random order."""
    E, O = emu(), refs.oracle()
    data = CM_CASES[CM_IDS.index("bwt_zipf_12k")][1][:5000]
    n = len(data)
    want = np.zeros(2 * n + 64, np.uint8)
    rw = O.orc_cm_encode(refs.ptr(data), n, refs.ptr(want))
    E.emu_set_schedule(schedule, 4242)
    try:
        got = np.zeros(2 * n + 64, np.uint8)
        assert E.emu_cm_encode(refs.ptr(data), n, refs.ptr(got)) == rw
        assert bytes(got[:rw]) == bytes(want[:rw])
        back = np.zeros(n + 8, np.uint8)
        E.emu_cm_decode(refs.ptr(want), rw, refs.ptr(back), n)
        assert bytes(back[:n]) == bytes(data)
    finally:
        E.emu_set_schedule(0, 1)


def _lzp_extra():
    rng = np.random.default_rng(5)
    rep = np.tile(rng.integers(0, 256, 700, dtype=np.uint8), 60)          # long matches, period 700
    runs = np.repeat(rng.integers(0, 3, 300, dtype=np.uint8), 150)        # every context repeats inside a window
    esc = rng.choice(np.array([0xF2, 0x41, 0x42], np.uint8), 30000)       # escape bytes with live slots
    mix = np.concatenate([rep[:9000], rng.integers(0, 256, 5000, dtype=np.uint8), rep[:9000], runs[:6000], esc[:4000]])
    return [("periodic_42k", rep), ("runs_45k", runs), ("escapes_30k", esc), ("mix_33k", mix)]


LZP_CASES = [(name, arr(d)) for name, d in synth.edge_cases()] + [
    ("source_96k", synth.source_corpus(96 << 10, seed=21)), ("log_64k", synth.log_stream(64 << 10, seed=22)),
    ("zipf_64k", synth.zipf_text(64 << 10, seed=23))] + _lzp_extra()


@pytest.mark.parametrize("name,data", LZP_CASES, ids=[c[0] for c in LZP_CASES])
def test_lzp_decode_kernel(name, data):
    E, O = emu(), refs.oracle()
    n = len(data)
    pad = np.zeros(n + 64, np.uint8)
    pad[:n] = data
    want = np.zeros(n + 64, np.uint8)
    got = np.zeros(n + 64, np.uint8)
    lut = np.zeros(1 << 18, np.int32)
    lp = lut.ctypes.data_as(refs.i32p)
    rw = O.orc_lzp_encode(refs.ptr(pad), n, refs.ptr(want), lp)
    if rw > 0:   # the encoder is covered by tests/test_emu_stages.py::test_lzp_scan_encoder
        for cut in (rw, rw - 1, rw // 2, 4, 3):
            cap = refs.bound(n)
            dw = np.zeros(cap + 64, np.uint8)
            dg = np.zeros(cap + 64, np.uint8)
            sw = O.orc_lzp_decode(refs.ptr(want), cut, refs.ptr(dw), cap, lp)
            lut_w = lut.copy()
            sg = E.emu_lzp_decode(refs.ptr(want), cut, refs.ptr(dg), cap, lp)
            assert sg == sw, (cut, sg, sw)
            if sw > 0:
                assert bytes(dg[:sg]) == bytes(dw[:sw])
                assert np.array_equal(lut, lut_w)   # same final table as the reference's
        # output capacity smaller than the decoded size: the copy is clamped like the reference's
        for cap in (n // 2, 5):
            if cap < 4:
                continue
            dw = np.zeros(n + 64, np.uint8)
            db = np.zeros(n + 64, np.uint8)
            sw = O.orc_lzp_decode(refs.ptr(want), rw, refs.ptr(dw), cap, lp)
            sb = E.emu_lzp_decode(refs.ptr(want), rw, refs.ptr(db), cap, lp)
            assert sb == sw, (cap, sb, sw)
            if sw > 0:
                assert bytes(db[:sb]) == bytes(dw[:sw])


def test_fuzz_small_inputs():
    """Random small inputs (several byte distributions) through the CM and LZP kernels."""
    E, O = emu(), refs.oracle()
    rng = np.random.default_rng(20260923)
    lut = np.zeros(1 << 18, np.int32)
    lp = lut.ctypes.data_as(refs.i32p)
    for it in range(40):
        n = int(rng.integers(1, 700))
        kind = it % 4
        if kind == 0:
            data = rng.integers(0, 256, n, dtype=np.uint8)
        elif kind == 1:
            data = rng.choice(np.array([0, 1, 255, 0xF2], np.uint8), n, p=[0.7, 0.1, 0.1, 0.1])
        elif kind == 2:
            data = np.repeat(rng.integers(0, 256, n // 7 + 1, dtype=np.uint8), 7)[:n]
        else:
            base = rng.integers(0, 256, max(n // 5, 1), dtype=np.uint8)
            data = np.tile(base, 6)[:n]
        data = np.ascontiguousarray(data)
        n = len(data)
        want = np.zeros(2 * n + 64, np.uint8)
        rw = O.orc_cm_encode(refs.ptr(data), n, refs.ptr(want))
        got = np.zeros(2 * n + 64, np.uint8)
        assert E.emu_cm_encode(refs.ptr(data), n, refs.ptr(got)) == rw, it
        assert bytes(got[:rw]) == bytes(want[:rw]), it
        cut = int(rng.integers(0, rw + 1))
        dw = np.zeros(n + 8, np.uint8)
        O.orc_cm_decode(refs.ptr(want), cut, refs.ptr(dw), n)
        back = np.zeros(n + 8, np.uint8)
        E.emu_cm_decode(refs.ptr(want), rw, refs.ptr(back), n)
        assert bytes(back[:n]) == bytes(data), it
        back = np.zeros(n + 8, np.uint8)
        E.emu_cm_decode(refs.ptr(want), cut, refs.ptr(back), n)
        assert bytes(back[:n]) == bytes(dw[:n]), (it, cut)
        # LZP on a longer, matchy input built from the same bytes
        long = np.ascontiguousarray(np.tile(data, 1 + 1200 // n)[:1200 + n])
        m = len(long)
        pad = np.zeros(m + 64, np.uint8)
        pad[:m] = long
        lw = np.zeros(m + 64, np.uint8)
        r0 = O.orc_lzp_encode(refs.ptr(pad), m, refs.ptr(lw), lp)
        if r0 > 0:
            cap = refs.bound(m)
            for cutl in (r0, int(rng.integers(0, r0 + 1))):
                d0 = np.zeros(cap + 64, np.uint8)
                s0 = O.orc_lzp_decode(refs.ptr(lw), cutl, refs.ptr(d0), cap, lp)
                for fn in (E.emu_lzp_decode,):
                    d1 = np.zeros(cap + 64, np.uint8)
                    assert fn(refs.ptr(lw), cutl, refs.ptr(d1), cap, lp) == s0, (it, cutl)
                    if s0 > 0:
                        assert bytes(d1[:s0]) == bytes(d0[:s0]), (it, cutl)
