"""Pins the CPU oracle (oracle/bz3_oracle.c) against
  (1) the reference's golden vector  examples/shakespeare.txt(.bz3)  (Makefile.am:81-83),
  (2) known answers computed by the compiled reference (SURVEY.md 8c / BASELINE.md section 2),
  (3) what the unmodified reference computes for the same inputs, stage by stage and block by block
      (tests/golden/reference_answers.json, written by tests/golden/make_reference_answers.py through the
      *_answer functions below).
CPU only."""
import ctypes as C
import hashlib
import os
import struct
from types import SimpleNamespace

import numpy as np
import pytest

from bzip3_b200 import synth
from tests import refs

O = refs.oracle()
CASES = synth.edge_cases()
IDS = [c[0] for c in CASES]
# the stage and block functions of the oracle; the reference's, with the same calling convention, are in
# tests/golden/make_reference_answers.py
ORACLE_STAGES = SimpleNamespace(crc=O.orc_crc32, mrle_encode=O.orc_mrle_encode, mrle_decode=O.orc_mrle_decode,
                                lzp_encode=O.orc_lzp_encode, lzp_decode=O.orc_lzp_decode, bwt=O.orc_bwt,
                                unbwt=O.orc_unbwt, cm_encode=O.orc_cm_encode, cm_decode=O.orc_cm_decode)
ORACLE_BLOCKS = SimpleNamespace(encode=refs.oracle_encode_block, decode=refs.oracle_decode_block)
HOSTILE = ["raw63", "coded65_text", "zeros_4k", "random_10k", "repeat_block_5000x20", "long_runs", "zipf_200k"]


def arr(b):
    return np.frombuffer(bytes(b), dtype=np.uint8).copy() if len(b) else np.zeros(1, np.uint8)[:0].copy()


def golden(name):
    with open(os.path.join(refs.GOLDEN, name), "rb") as f:
        return f.read()


# ------------------------------------------------------------------ golden vectors / KATs
def parse_cli_stream(blob):
    """bzip3 CLI container (src/main.c:174-179, :249-253): 'BZ3v1' u32 block_size, then [csize][osize][payload]*"""
    assert blob[:5] == b"BZ3v1"
    bs = struct.unpack("<I", blob[5:9])[0]
    at, blocks = 9, []
    while at < len(blob):
        cs, osz = struct.unpack("<ii", blob[at:at + 8])
        blocks.append((blob[at + 8:at + 8 + cs], osz))
        at += 8 + cs
    return bs, blocks


def test_golden_decode_shakespeare():
    bs, blocks = parse_cli_stream(golden("shakespeare.txt.bz3"))
    assert bs == 4 << 20 and len(blocks) == 2
    plain = b""
    for enc, osz in blocks:
        out, r, e = refs.oracle_decode_block(enc, osz, bs)
        assert r == osz and e == 0
        plain += out
    assert plain == golden("shakespeare.txt")


def test_kat_encode_shakespeare_b8():
    # computed by the compiled reference: bzip3 -e -b 8 examples/shakespeare.txt (BASELINE.md section 2)
    data = golden("shakespeare.txt")
    enc, r, e = refs.oracle_encode_block(data, 8 << 20)
    assert e == 0 and r == 1229797
    crc, idx, model, lzp = struct.unpack("<IiBi", enc[:13])
    assert (crc, idx, model, lzp) == (0x18A1405E, 1980452, 2, 5314513)
    stream = b"BZ3v1" + struct.pack("<I", 8 << 20) + struct.pack("<ii", r, len(data)) + enc
    assert len(stream) == 1229814
    assert hashlib.sha256(stream).hexdigest() == "6ed262b586d6e58aa00429ac1776b3ca29ca59283c2008f43378fef87755cee6"


def test_crc_known_values():
    assert O.orc_crc32(1, refs.ptr(arr(b"")), 0) == 1
    d = arr(golden("shakespeare.txt"))
    assert O.orc_crc32(1, refs.ptr(d), len(d)) == 0x18A1405E


@pytest.mark.parametrize("name", ["63_byte_file.bin", "65_byte_file.bin"])
def test_seed_files_roundtrip(name):
    data = golden(name)
    enc, r, e = refs.oracle_encode_block(data, 65 * 1024)
    assert r > 0
    if len(data) < 64:
        assert r == len(data) + 8 and struct.unpack("<i", enc[4:8])[0] == -1
    out, r2, e2 = refs.oracle_decode_block(enc, len(data), 65 * 1024)
    assert out == data


# ------------------------------------------------------------------ stage-level differential vs the reference
# Each *_answer function runs one comparison on one implementation and returns what it saw: return values and digests
# of the bytes written.  The tests take the oracle's; the stored answers are the reference's, through the same function.
def crc_answer(S, data):
    a = arr(data)
    return S.crc(1, refs.ptr(a), len(a))


def mrle_answer(S, data):
    """mRLE encode, then decodes of the whole encoding and of truncated ones: the failure flag and the bytes produced
    must agree too."""
    a = arr(data)
    n = len(a)
    o = np.zeros(2 * n + 64, np.uint8)
    r = S.mrle_encode(refs.ptr(a.copy()), n, refs.ptr(o))
    out = [r, refs.digest(o[:r])]
    for cut in (r, r - 1, r // 2, 33, 32, 31):
        if cut < 0:
            continue
        d = np.zeros(n + 8, np.uint8)
        e = S.mrle_decode(refs.ptr(o), refs.ptr(d), n, cut)
        out.append([cut, e, refs.digest(d[:n] if cut == r else d)])
    return out


def lzp_answer(S, data):
    """LZP encode, then decodes of the whole encoding and of truncated ones with the same table."""
    a = arr(data)
    n = len(a)
    pad = np.zeros(n + 64, np.uint8)
    pad[:n] = a
    o = np.zeros(n + 64, np.uint8)
    lut = np.zeros(1 << 18, np.int32)
    lp = lut.ctypes.data_as(refs.i32p)
    r = S.lzp_encode(refs.ptr(pad), n, refs.ptr(o), lp)
    out = [r]
    if r > 0:
        out.append(refs.digest(o[:r]))
        cap = refs.bound(n) + 64
        for cut in (r, r - 1, r - 2, r // 2, 5, 4, 3):
            if cut < 0:
                continue
            d = np.zeros(cap, np.uint8)
            s = S.lzp_decode(refs.ptr(o), cut, refs.ptr(d), refs.bound(n), lp)
            out.append([cut, s, refs.digest(d[:s]) if s > 0 else None])
    return out


def bwt_answer(S, data):
    """BWT, its inverse, and the inverse with primary indices out of range."""
    a = arr(data)
    n = len(a)
    u = np.zeros(n + 8, np.uint8)
    i = S.bwt(refs.ptr(a), refs.ptr(u), n)
    t = np.zeros(n + 8, np.uint8)
    out = [i, refs.digest(u[:n]), S.unbwt(refs.ptr(u), refs.ptr(t), n, i), refs.digest(t[:n])]
    if n >= 2:
        out.append([S.unbwt(refs.ptr(u), refs.ptr(t), n, bad) for bad in (0, -3, n + 1)])
    return out


def cm_answer(S, data):
    """CM encode, then decodes of the whole payload and of truncated ones (read as 0xFF.. like read_in)."""
    a = arr(data)
    n = len(a)
    o = np.zeros(2 * n + 64, np.uint8)
    r = S.cm_encode(refs.ptr(a.copy()), n, refs.ptr(o))
    out = [r, refs.digest(o[:r])]
    for insize in (r, max(r - 3, 0), r // 2, 0):
        d = np.zeros(n + 8, np.uint8)
        S.cm_decode(refs.ptr(o), insize, refs.ptr(d), n)
        out.append([insize, refs.digest(d)])
    return out


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_crc(name, data):
    refs.check_answer(f"stage_crc/{name}", crc_answer(ORACLE_STAGES, data))


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_mrle(name, data):
    got = mrle_answer(ORACLE_STAGES, data)
    refs.check_answer(f"stage_mrle/{name}", got)
    assert got[2][1:] == [0, refs.digest(data)]


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_lzp(name, data):
    got = lzp_answer(ORACLE_STAGES, data)
    refs.check_answer(f"stage_lzp/{name}", got)
    if got[0] > 0:
        assert got[2][1:] == [len(data), refs.digest(data)]


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_bwt(name, data):
    got = bwt_answer(ORACLE_STAGES, data)
    refs.check_answer(f"stage_bwt/{name}", got)
    assert got[2:4] == [0, refs.digest(data)]


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_stage_cm(name, data):
    got = cm_answer(ORACLE_STAGES, data)
    refs.check_answer(f"stage_cm/{name}", got)
    assert got[2][1] == refs.digest(data + bytes(8))


# ------------------------------------------------------------------ block-level differential
def block_answer(B, data):
    bs = max(65 * 1024, len(data))
    enc, r, e = B.encode(data, bs)
    dec, d, de = B.decode(enc, len(data), bs)
    return [r, e, refs.digest(enc), d, de, refs.digest(dec)]


@pytest.mark.parametrize("name,data", CASES, ids=IDS)
def test_block_encode_decode_vs_reference(name, data):
    got = block_answer(ORACLE_BLOCKS, data)
    refs.check_answer(f"block/{name}", got)
    assert got[3:] == [len(data), 0, refs.digest(data)]


def test_block_too_big():
    got = list(refs.oracle_encode_block(bytes(70000), 65 * 1024)[1:])
    refs.check_answer("block_too_big", got)
    assert got == [-1, -6]


def hostile_variants(enc, osz, bs, rng):
    """(enc, orig_size, buffer_size, compressed_size) tuples in the spirit of examples/fuzz-decode-block.c:173-207."""
    out = [(enc, osz, None, None), (enc, osz + 1, None, None), (enc, max(osz - 1, 0), None, None),
           (enc, osz, 8, None), (enc, osz, len(enc) - 1, None), (enc, osz, None, -5), (enc, osz, None, 4),
           (enc, -1, None, None), (enc, refs.bound(bs) + 1, None, None), (enc, osz, osz, None),
           (enc[:len(enc) // 2], osz, None, None), (enc[:9], osz, None, None), (enc[:12], osz, None, None)]
    for _ in range(12):
        b = bytearray(enc)
        k = int(rng.integers(0, len(b)))
        b[k] ^= 1 << int(rng.integers(0, 8))
        out.append((bytes(b), osz, None, None))
    for field in (4, 8, 9, 13):  # bwt index, model byte, size fields
        if len(enc) > field + 4:
            for v in (0, 1, 0x7FFFFFFF, 0xFFFFFFFE, osz + 7):
                b = bytearray(enc)
                if field == 8:
                    b[8] = v & 0xFF
                else:
                    b[field:field + 4] = struct.pack("<I", v & 0xFFFFFFFF)
                out.append((bytes(b), osz, None, None))
    return out


def hostile_answer(B, name):
    """Return value, error number and bytes of decodes of damaged encodings of one of the CASES."""
    data = dict(CASES)[name]
    bs = max(65 * 1024, len(data))
    enc = B.encode(data, bs)[0]
    rng = np.random.default_rng(len(data))
    out = []
    for venc, osz, bsz, csz in hostile_variants(enc, len(data), bs, rng):
        dec, r, e = B.decode(venc, osz, bs, buffer_size=bsz, compressed_size=csz)
        out.append([r, e, refs.digest(dec) if r >= 0 else None])
    return out


@pytest.mark.parametrize("name", HOSTILE)
def test_hostile_decode_error_parity(name):
    refs.check_answer(f"hostile/{name}", hostile_answer(ORACLE_BLOCKS, name))


def medium_corpora():
    return [synth.zipf_text(1_500_000).tobytes(), synth.source_corpus(1_500_000).tobytes(),
            synth.mixed(1_200_000, segment=300_000).tobytes(), synth.log_stream(800_000).tobytes()]


def medium_answer(B, datas):
    bs = 2 << 20
    out = []
    for data in datas:
        enc, r, e = B.encode(data, bs)
        out.append([r, e, refs.digest(enc)])
    return out


def test_medium_corpora_block_parity():
    datas = medium_corpora()
    refs.check_answer("medium_corpora", medium_answer(ORACLE_BLOCKS, datas))
    for data in datas:
        assert refs.oracle_decode_block(refs.oracle_encode_block(data, 2 << 20)[0], len(data), 2 << 20)[0] == data
