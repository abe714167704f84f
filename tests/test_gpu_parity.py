"""GPU parity tests: every stage kernel and the whole block codec, called through the C ABI of
libbzip3_b200.so, against the CPU oracle (oracle/bz3_oracle.c), the committed golden vectors and
known answers of the reference.  Bit-exact: all arithmetic on this path is integer."""
import ctypes as C
import hashlib
import os
import struct

import numpy as np
import pytest

import bzip3_b200
from bzip3_b200 import synth
from tests import refs
from tests.test_oracle import hostile_variants, parse_cli_stream

pytestmark = pytest.mark.gpu

CASES = synth.edge_cases()
IDS = [c[0] for c in CASES]
BS = 1 << 20


def arr(b):
    return np.frombuffer(bytes(b), dtype=np.uint8).copy()


def first_diff(a, b):
    a = np.frombuffer(a, np.uint8)
    b = np.frombuffer(b, np.uint8)
    n = min(len(a), len(b))
    d = np.nonzero(a[:n] != b[:n])[0]
    return (int(d[0]) if len(d) else n, len(a), len(b))


@pytest.fixture(scope="module")
def st():
    with bzip3_b200.Bz3State(BS) as s:
        yield s


@pytest.fixture(scope="module")
def O():
    return refs.oracle()


def golden(name):
    with open(os.path.join(refs.GOLDEN, name), "rb") as f:
        return f.read()


# ---------------------------------------------------------------- stages
@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_crc(st, O, name, data):
    a = arr(data)
    pad = np.zeros(len(a) + 16, np.uint8)
    pad[:len(a)] = a
    assert st.L.bz3_b200_stage_crc(st.handle, refs.ptr(pad), len(a)) == O.orc_crc32(1, refs.ptr(pad), len(a))


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_rle(st, O, name, data):
    a = arr(data)
    n = len(a)
    pad = np.zeros(n + 16, np.uint8)
    pad[:n] = a
    want = np.zeros(2 * n + 64, np.uint8)
    got = np.zeros(2 * n + 64, np.uint8)
    rw = O.orc_mrle_encode(refs.ptr(pad), n, refs.ptr(want))
    rg = st.L.bz3_b200_stage_rle_encode(st.handle, refs.ptr(pad), n, refs.ptr(got))
    assert rg == rw, (rg, rw)
    assert bytes(got[:rg]) == bytes(want[:rw]), first_diff(got[:rg], want[:rw])
    for cut in (rw, rw - 1, rw // 2, 33, 32, 31):
        if cut < 0:
            continue
        dw = np.zeros(n + 8, np.uint8)
        dg = np.zeros(n + 8, np.uint8)
        ew = O.orc_mrle_decode(refs.ptr(want), refs.ptr(dw), n, cut)
        eg = st.L.bz3_b200_stage_rle_decode(st.handle, refs.ptr(want), cut, refs.ptr(dg), n)
        assert eg == ew, (cut, eg, ew)
        assert bytes(dg[:n]) == bytes(dw[:n]), (cut, first_diff(dg[:n], dw[:n]))


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_lzp(st, O, name, data):
    _check_lzp(st, O, data)


def _check_lzp(st, O, data):
    a = arr(data)
    n = len(a)
    pad = np.zeros(n + 64, np.uint8)
    pad[:n] = a
    want = np.zeros(n + 64, np.uint8)
    got = np.zeros(n + 64, np.uint8)
    lut = np.zeros(1 << 18, np.int32)
    lp = lut.ctypes.data_as(refs.i32p)
    rw = O.orc_lzp_encode(refs.ptr(pad), n, refs.ptr(want), lp)
    rg = st.L.bz3_b200_stage_lzp_encode(st.handle, refs.ptr(pad), n, refs.ptr(got))
    assert rg == rw
    if rw > 0:
        assert bytes(got[:rg]) == bytes(want[:rw]), first_diff(got[:rg], want[:rw])
        for cut in (rw, rw - 1, rw // 2, 4, 3):
            cap = refs.bound(n)
            dw = np.zeros(cap + 64, np.uint8)
            dg = np.zeros(cap + 64, np.uint8)
            sw = O.orc_lzp_decode(refs.ptr(want), cut, refs.ptr(dw), cap, lp)
            sg = st.L.bz3_b200_stage_lzp_decode(st.handle, refs.ptr(want), cut, refs.ptr(dg), cap)
            assert sg == sw, (cut, sg, sw)
            if sw > 0:
                assert bytes(dg[:sg]) == bytes(dw[:sw]), (cut, first_diff(dg[:sg], dw[:sw]))


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_bwt(st, O, name, data):
    a = arr(data)
    n = len(a)
    pad = np.zeros(n + 16, np.uint8)
    pad[:n] = a
    want = np.zeros(n + 8, np.uint8)
    got = np.zeros(n + 8, np.uint8)
    iw = O.orc_bwt(refs.ptr(pad), refs.ptr(want), n)
    ig = st.L.bz3_b200_stage_bwt(st.handle, refs.ptr(pad), n, refs.ptr(got))
    assert ig == iw, (ig, iw)
    assert bytes(got[:n]) == bytes(want[:n]), first_diff(got[:n], want[:n])
    if n >= 2:
        back = np.zeros(n + 8, np.uint8)
        assert st.L.bz3_b200_stage_unbwt(st.handle, refs.ptr(want), n, iw, refs.ptr(back)) == 0
        assert bytes(back[:n]) == bytes(a), first_diff(back[:n], a)
        for bad in (0, -2, n + 1):
            assert st.L.bz3_b200_stage_unbwt(st.handle, refs.ptr(want), n, bad, refs.ptr(back)) == -1


def test_stage_unbwt_on_garbage_matches_reference_semantics(st, O):
    """Corrupt transforms: the walk leaves the text path early; output must equal the oracle's restatement
    of what libsais emits (checked against the reference itself in tests/test_oracle.py)."""
    rng = np.random.default_rng(7)
    for t in range(120):
        n = int(rng.integers(2, 3000)) if t % 4 else int(rng.integers(2, 16))
        k = int(rng.integers(1, 5)) if t % 2 else 256
        L = rng.integers(0, k, n).astype(np.uint8)
        idx = int(rng.integers(1, n + 1))
        want = np.zeros(n + 8, np.uint8)
        got = np.zeros(n + 8, np.uint8)
        assert O.orc_unbwt(refs.ptr(L), refs.ptr(want), n, idx) == 0
        assert st.L.bz3_b200_stage_unbwt(st.handle, refs.ptr(L), n, idx, refs.ptr(got)) == 0
        assert bytes(got[:n]) == bytes(want[:n]), (t, n, k, idx, first_diff(got[:n], want[:n]))


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_cm(st, O, name, data):
    a = arr(data)
    n = len(a)
    pad = np.zeros(n + 16, np.uint8)
    pad[:n] = a
    want = np.zeros(2 * n + 64, np.uint8)
    got = np.zeros(2 * n + 64, np.uint8)
    rw = O.orc_cm_encode(refs.ptr(pad), n, refs.ptr(want))
    rg = st.L.bz3_b200_stage_cm_encode(st.handle, refs.ptr(pad), n, refs.ptr(got))
    assert rg == rw, (rg, rw)
    assert bytes(got[:rg]) == bytes(want[:rw]), first_diff(got[:rg], want[:rw])
    for insize in (rw, max(rw - 3, 0), rw // 2):   # whole stream and truncated ones (read_in() past the end, :345)
        dw = np.zeros(n + 8, np.uint8)
        dg = np.zeros(n + 8, np.uint8)
        O.orc_cm_decode(refs.ptr(want), insize, refs.ptr(dw), n)
        assert st.L.bz3_b200_stage_cm_decode(st.handle, refs.ptr(want), insize, refs.ptr(dg), n) == 0
        assert bytes(dg[:n]) == bytes(dw[:n]), (insize, first_diff(dg[:n], dw[:n]))


def test_stage_cm_exhausted_streams(st, O):
    """Payloads that end early or are garbage, decoded far past their end (read_in() feeds -1, src/libbz3.c:345):
    the decoder's shortcuts must be off once the stream is exhausted.  Same cases as the emulator test."""
    rng = np.random.default_rng(31337)
    base = arr(synth.zipf_text(64 << 10, seed=7))
    n = 20000
    bw = np.zeros(n + 16, np.uint8)
    O.orc_bwt(refs.ptr(base[:n].copy()), refs.ptr(bw), n)
    enc = np.zeros(2 * n + 64, np.uint8)
    r = O.orc_cm_encode(refs.ptr(bw), n, refs.ptr(enc))
    payloads = [(enc, cut) for cut in list(range(0, 12)) + [r // 7, r // 3, r - 9, r - 5, r - 4, r - 2, r - 1]]
    for k in range(40):
        g = np.zeros(64, np.uint8)
        m = int(rng.integers(1, 40))
        g[:m] = rng.integers(0, 256, m, dtype=np.uint8) if k % 3 else np.full(m, 255 * (k % 2), np.uint8)
        payloads.append((g, m))
    for buf, insize in payloads:
        dw = np.zeros(n + 8, np.uint8)
        dg = np.zeros(n + 8, np.uint8)
        O.orc_cm_decode(refs.ptr(buf), insize, refs.ptr(dw), n)
        assert st.L.bz3_b200_stage_cm_decode(st.handle, refs.ptr(buf), insize, refs.ptr(dg), n) == 0
        assert bytes(dg[:n]) == bytes(dw[:n]), (insize, first_diff(dg[:n], dw[:n]))


# ---------------------------------------------------------------- whole blocks
@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_block_roundtrip_vs_oracle(st, name, data):
    enc_o, r_o, e_o = refs.oracle_encode_block(data, BS)
    enc_g, r_g = st.encode_block(data)
    assert r_g == r_o, (r_g, r_o, st.last_error)
    if len(data) >= 64:
        assert st.last_error == e_o
    assert enc_g == enc_o, first_diff(enc_g, enc_o)
    dec, r = st.decode_block(enc_o, len(data))
    assert r == len(data) and dec == data
    if len(data) >= 64:
        assert st.last_error == 0


def test_block_too_big(st):
    enc, r = st.encode_block(bytes(BS + 1))
    assert r == -1 and st.last_error == bzip3_b200.BZ3_ERR_DATA_TOO_BIG


def test_last_error_untouched_on_raw_paths(st):
    st.encode_block(bytes(BS + 1))
    assert st.last_error == bzip3_b200.BZ3_ERR_DATA_TOO_BIG
    enc, r = st.encode_block(b"tiny")  # reference returns early without touching last_error (src/libbz3.c:596-601)
    assert r == 12 and st.last_error == bzip3_b200.BZ3_ERR_DATA_TOO_BIG
    dec, r = st.decode_block(enc, 4)
    assert dec == b"tiny" and st.last_error == bzip3_b200.BZ3_ERR_DATA_TOO_BIG


@pytest.mark.parametrize("name", ["raw63", "coded65_text", "zeros_4k", "random_10k", "repeat_block_5000x20",
                                  "long_runs", "zipf_200k"])
def test_hostile_decode_error_parity(st, name):
    data = dict(CASES)[name]
    enc, r, e = refs.oracle_encode_block(data, BS)
    rng = np.random.default_rng(len(data))
    for k, (venc, osz, bsz, csz) in enumerate(hostile_variants(enc, len(data), BS, rng)):
        want = refs.oracle_decode_block(venc, osz, BS, buffer_size=bsz, compressed_size=csz, err_init=55)
        # same starting last_error on our side: provoke a known state first
        st.L.bz3_b200_stats_reset(st.handle)
        got_bytes, got_r = st.decode_block(venc, osz, buffer_size=bsz, compressed_size=csz)
        assert got_r == want[1], (name, k, got_r, want[1:], st.last_error)
        if want[2] != 55:  # the oracle wrote an error code
            assert st.last_error == want[2], (name, k, st.last_error, want[2])
        if got_r >= 0:
            assert got_bytes == want[0]


def test_golden_shakespeare_decode_and_kat_encode():
    plain = golden("shakespeare.txt")
    bs, blocks = parse_cli_stream(golden("shakespeare.txt.bz3"))
    with bzip3_b200.Bz3State(bs) as s:
        out = b""
        for enc, osz in blocks:
            dec, r = s.decode_block(enc, osz)
            assert r == osz and s.last_error == 0
            out += dec
        assert out == plain
    with bzip3_b200.Bz3State(8 << 20) as s:
        enc, r = s.encode_block(plain)
        assert r == 1229797 and s.last_error == 0
        stream = b"BZ3v1" + struct.pack("<I", 8 << 20) + struct.pack("<ii", r, len(plain)) + enc
        assert hashlib.sha256(stream).hexdigest() == "6ed262b586d6e58aa00429ac1776b3ca29ca59283c2008f43378fef87755cee6"
        dec, r2 = s.decode_block(enc, len(plain))
        assert dec == plain


def test_batch_api_matches_single_blocks():
    rng = np.random.default_rng(3)
    datas = [synth.zipf_text(300_000, seed=5).tobytes(), synth.log_stream(200_000, seed=6).tobytes(),
             bytes(rng.integers(0, 256, 100_000, dtype=np.uint8)), b"short", synth.source_corpus(400_000, seed=8).tobytes()]
    bs = 1 << 19
    states = [bzip3_b200.Bz3State(bs) for _ in datas]
    try:
        bufs = []
        for d in datas:
            b = np.zeros(bzip3_b200.bound(bs) + 64, np.uint8)
            b[:len(d)] = np.frombuffer(d, np.uint8)
            bufs.append(b)
        sizes = bzip3_b200.encode_blocks(states, bufs, [len(d) for d in datas])
        for d, b, sz, s in zip(datas, bufs, sizes, states):
            want = refs.oracle_encode_block(d, bs)
            assert sz == want[1] and bytes(b[:sz]) == want[0]
        errs = bzip3_b200.decode_blocks(states, bufs, [len(b) for b in bufs], sizes, [len(d) for d in datas])
        for d, b, e in zip(datas, bufs, errs):
            assert bytes(b[:len(d)]) == d
    finally:
        for s in states:
            s.close()


def test_frame_api_roundtrip():
    L = bzip3_b200.lib()
    data = synth.zipf_text(300_000, seed=11)
    out = np.zeros(bzip3_b200.bound(len(data)) + 64, np.uint8)
    osz = C.c_size_t(len(out))
    assert L.bz3_compress(1 << 17, refs.ptr(data), refs.ptr(out), len(data), C.byref(osz)) == 0
    back = np.zeros(len(data) + 64, np.uint8)
    bsz = C.c_size_t(len(back))
    assert L.bz3_decompress(refs.ptr(out), refs.ptr(back), osz.value, C.byref(bsz)) == 0
    assert bsz.value == len(data) and bytes(back[:len(data)]) == data.tobytes()
    # the frame the reference's bz3_compress writes
    refs.check_answer("frame/zipf300k_seed11_b128k", [osz.value, refs.digest(out[:osz.value])])


def test_medium_corpora_block_parity():
    bs = 4 << 20
    with bzip3_b200.Bz3State(bs) as s:
        for gen, n in ((synth.zipf_text, 3_000_000), (synth.source_corpus, 3_000_000), (synth.log_stream, 1_500_000)):
            data = gen(n).tobytes()
            want = refs.oracle_encode_block(data, bs)
            enc, r = s.encode_block(data)
            assert r == want[1] and enc == want[0], first_diff(enc or b"", want[0])
            dec, r2 = s.decode_block(enc, len(data))
            assert dec == data
        mixed = synth.mixed(2_000_000, segment=400_000).tobytes()
        want = refs.oracle_encode_block(mixed, bs)
        enc, r = s.encode_block(mixed)
        assert enc == want[0]


def test_reference_cross_decode_when_available():
    """The block equals the reference's bz3_encode_block output (stored answer; the reference decodes it to the input
    where the answer was made), and decodes here."""
    data = synth.zipf_text(500_000, seed=21).tobytes()
    with bzip3_b200.Bz3State(1 << 20) as s:
        enc, r = s.encode_block(data)
        refs.check_answer("cross/zipf500k_seed21_b1m", [r, s.last_error, refs.digest(enc)])
        assert s.decode_block(enc, len(data))[0] == data
